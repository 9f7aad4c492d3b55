#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused drone-navigation control step on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): step-only throughput, 4096 CF2X envs per GPU, DYN physics,
240 Hz physics / 30 Hz control (S = 8 substeps fused per launch), circle track, THRUST actions with
normalize_actions, 13-dim observation, default reward, pre-generated saturating U(-1,1) actions
(reset-heavy).  One "step" = one launch of the fused kernel over the whole batch.

Printed JSON line (rank 0): see the task contract.  Extra keys:
  value            device-timed, inputs resident in HBM, L2 flushed between the timed launches
  l2_resident      same workload replayed back to back from a CUDA graph (state stays in the 126 MB L2,
                   as it does in real use at this batch size) -- launch-latency regime
  sweep            larger batches (65 536 / 1 Mi / 4 Mi envs): the HBM regime, with roofline fractions
  roofline         dominant kernel (step_kernel) at the headline workload
  roofline_hbm     the same kernel at the largest swept batch (state + outputs >> L2)
  e2e              the same metric through the C-ABI host-buffer call (dn_step_host): pinned host
                   actions -> H2D -> kernel -> D2H obs/reward/done/found every step
  cpu_baseline     the CPU oracle (numpy port of the reference step) on the host cores, bounded sample
  cpu_baseline_batched  best-case CPU: the same algorithm as array operations over all envs at once
                   (oracle/batched_oracle.py), one process per host core -- not how the reference runs
`--impl reference` times that CPU path as its own arm (the reference is pure Python; pybullet / SB3 are
not installable here, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "env-steps/sec (fused substeps)"
UNIT = "env-steps/s"
BYTES_PER_ENV_STEP = 16 + 112 + 112 + 52 + 4 + 1 + 4   # action | state in | state out | obs | reward | done | found  (DESIGN.md)
HOVER = 0.092227
DUMP_LIMIT = 64 << 20                   # bytes, all files of --dump-outputs together


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """--dump-outputs: each [N, ...] array of `arrays` as out_dir/<name>.npy, float32 kept, every other dtype as float64
    (exact for the integer outputs).  If they would take more than `limit` bytes together, the same fixed, seeded sample
    of rows is written of each, and the sampled row numbers as env_index.npy."""
    arrays = {k: np.asarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > limit - 4096:                    # 4 KiB for the .npy headers
        rows = (limit - 4096) // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, size=rows, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def track_setup(track: str):
    from drl_dronenavigation_b200 import Track, Waypoints, track_targets
    if track == "circle":
        tr = Track(Waypoints.circle(radius=1, num_points=6, height=1), circle=True)
    else:
        tr = Track(Waypoints.reaching(), circle=False)
    return np.array(track_targets(tr)), np.array(tr.initial_xyzs, dtype=np.float64), np.array(tr.aviary_dim), tr.is_circle


# ----------------------------------------------------------------------------------------------
# clocks sampler (recipe line of /opt/skills/guides/B200_PROFILING.md)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.15 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:   # timed region shorter than one sample: take whatever was seen
            for ts, line in self.rows:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); smax = float(f[2])
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle (numpy port of the reference step), one env object per worker process slot,
# exactly like SubprocVecEnv workers
# ----------------------------------------------------------------------------------------------
def _cpu_worker(args):
    track, S, n_envs, n_steps, seed = args
    from oracle.dyn_oracle import OracleWorker, make_reference_env
    ws = [OracleWorker(make_reference_env(track, pyb_freq=240, ctrl_freq=240 // S), normalize_obs=False) for _ in range(n_envs)]
    for w in ws:
        w.reset()
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, size=(n_steps, n_envs, 4)).astype(np.float32)
    t0 = time.perf_counter()
    for t in range(n_steps):
        for i, w in enumerate(ws):
            w.step(acts[t, i])
    return time.perf_counter() - t0


def cpu_oracle_rate(track, S, envs_per_proc, steps, procs):
    """env-steps/s of the numpy oracle over `procs` processes (sum of per-process rates by max time)."""
    with mp.get_context("fork").Pool(procs) as pool:
        times = pool.map(_cpu_worker, [(track, S, envs_per_proc, steps, 100 + p) for p in range(procs)])
    return procs * envs_per_proc * steps / max(times), max(times)


def cpu_baseline(track, S, budget_s=12.0):
    cores = os.cpu_count() or 1
    rate1, _ = cpu_oracle_rate(track, S, 2, 40, cores)                       # calibration
    steps = max(20, int(budget_s * rate1 / (cores * 4)))
    rate, dt = cpu_oracle_rate(track, S, 4, steps, cores)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"numpy oracle (FP64 port of PBDroneEnv.step + BaseAviary._dynamics), {cores} processes x 4 envs x {steps} "
                      f"control steps, S={S}, {track} track, saturating actions, {dt:.1f} s"}


def _cpu_batched_worker(args):
    track, S, n_envs, n_steps, seed = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    from oracle.batched_oracle import BatchedOracle
    B = BatchedOracle(n_envs, track, pyb_freq=240, ctrl_freq=240 // S)
    acts = np.random.default_rng(seed).uniform(-1, 1, size=(n_steps + 1, n_envs, 4)).astype(np.float32)
    B.step(acts[0])
    t0 = time.perf_counter()
    for t in range(n_steps):
        B.step(acts[t + 1])
    return time.perf_counter() - t0


def cpu_baseline_batched(track, S, envs, budget_s=10.0):
    """Best-case CPU figure (SURVEY 8d): the batched numpy oracle, one replica of the workload's batch per host core
    (splitting the batch over the cores instead leaves each process dominated by the interpreter: 3.6e5 vs 1e6 here)."""
    cores = os.cpu_count() or 1
    per = max(1, envs)
    with mp.get_context("fork").Pool(cores) as pool:
        t1 = max(pool.map(_cpu_batched_worker, [(track, S, per, 2, 50 + p) for p in range(cores)])) / 2      # calibration
        steps = int(max(3, min(200, budget_s / max(t1, 1e-6))))
        times = pool.map(_cpu_batched_worker, [(track, S, per, steps, 100 + p) for p in range(cores)])
    return {"value": cores * per * steps / max(times), "unit": UNIT, "cores": cores, "kind": "port (batched numpy)",
            "sample": f"oracle/batched_oracle.py, {cores} processes x {per} envs x {steps} control steps, S={S}, {track} track, "
                      f"saturating actions, {max(times):.1f} s; the reference itself steps one Python env per worker process"}


def pybullet_cpu():
    """SURVEY 8d (ii): the reference's real PyBullet path can only be timed if its third-party stack imports."""
    missing = []
    for mod in ("pybullet", "gymnasium", "stable_baselines3"):
        try:
            __import__(mod)
        except Exception:  # noqa: BLE001
            missing.append(mod)
    if missing:
        return "n/a (not installable: " + ", ".join(missing) + " missing on this box, no network, no wheel)"
    return "n/a (modules import, but /root/reference is not present on the GPU box)"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is pure Python on
    PyBullet; neither pybullet nor gymnasium nor SB3 is installable here, and its own DYN branch is dead
    code, so the arm times the oracle port of it with every host core, SubprocVecEnv-style."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    S, track = args.substeps, args.track
    cores = os.cpu_count() or 1
    K, W = args.steps, args.warmup
    rate1, _ = cpu_oracle_rate(track, S, 2, 20, cores)
    budget = 120.0
    envs_per_proc = int(max(1, min(args.envs // cores, budget * rate1 / (cores * (K + W)))))
    n_envs = envs_per_proc * cores
    # one "step" = one control step of a bounded sample of the workload's envs (n_envs of args.envs)
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_cpu_worker, [(track, S, envs_per_proc, max(W, 1), 7 + p) for p in range(cores)])          # warm-up
        t0 = time.perf_counter()
        times = pool.map(_cpu_worker, [(track, S, envs_per_proc, K, 100 + p) for p in range(cores)])
        wall = time.perf_counter() - t0
    value = n_envs * K / max(times)
    sample = (f"{n_envs} of {args.envs} envs ({cores} processes x {envs_per_proc}), {K} control steps, S={S}, numpy oracle port "
              f"of the reference step (pybullet/SB3 not installable; reference DYN branch is dead code)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * max(times) / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": bench_config(args, int(os.environ.get("WORLD_SIZE", "1"))), "envs_in_sample": n_envs,
            "pybullet_cpu": pybullet_cpu(),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": wall}
    print(json.dumps(line), flush=True)


def bench_config(args, world):
    """The `config` object of BOTH arms (the reference arm runs "on your arm's config"): identical keys and values."""
    return {"workload": workload_name(args), "envs_per_gpu": args.envs, "substeps": args.substeps, "track": args.track,
            "actions": args.actions, "l2": "inputs larger than L2 (rotating handles, no flush kernel)",
            "parallelism": f"env-shard x{world} (no data-path collective)"}


def workload_name(args):
    return (f"step-only throughput: {args.envs} CF2X envs per GPU, Physics.DYN, 240 Hz physics / {240 // args.substeps} Hz control "
            f"(S={args.substeps}), {args.track} track, THRUST+normalize_actions, obs13, default reward, {args.actions} actions")


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def make_env(n_envs, args, device, env_id_offset=0, **kw):
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    targets, init, dim, is_circle = track_setup(args.track)
    return BatchedDroneEnv(n_envs, targets, threshold=0.3, discount=0.999, max_steps=4096, aviary_dim=dim,
                           initial_xyzs=init, pyb_freq=240, ctrl_freq=240 // args.substeps, cylinder=True, circle=is_circle,
                           include_distance=True, normalize_actions=True, device=device, env_id_offset=env_id_offset, **kw)


def baseline_configs(args, dev, K):
    """Step-only throughput of the fused kernel on the env shape of every BASELINE.json config (SURVEY 8d table), one
    GPU's share each, replayed from CUDA graphs (no host launch cost; working sets below 126 MB stay in L2, as they do
    in real use at these sizes).  The headline `value` above is config 2 measured the strict way (L2 flushed, per-launch
    events); these lines are context for the other four and are NOT headline numbers."""
    import copy
    import torch
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200 import _lib as L
    specs = [
        (1, "README PPO run: 12 envs, 240/240 Hz, circle, per-env NormalizeObservation", 12, 1, "circle", dict(normalize_obs=True)),
        (2, "4096 envs, 240/30 Hz, circle", 4096, 8, "circle", {}),
        (3, "65536 envs per GPU, 240/30 Hz, reaching track (segment tube)", 65536, 8, "reaching", {}),
        (4, "16384 envs, 240/30 Hz, circle, drag + ground effect", 16384, 8, "circle", dict(physics=Physics.PYB_GND_DRAG_DW)),
    ] + [(5, f"131072 envs per GPU (1 Mi / 8), 240/30 Hz, circle, reward_id={rid}", 131072, 8, "circle", dict(reward_id=rid))
         for rid in (L.DN_REWARD_DEFAULT, L.DN_REWARD_DUMMY, L.DN_REWARD_THRUSTENV, L.DN_REWARD_HER, L.DN_REWARD_REACHING, L.DN_REWARD_PROGRESS,
                     L.DN_REWARD_HOVER, L.DN_REWARD_FLYTHRUGATE, L.DN_REWARD_BOOTSTRAPPED, L.DN_REWARD_CHAMP)]
    out = []
    for cid, name, n, S, track, kw in specs:
        try:
            a = copy.copy(args); a.substeps, a.track = S, track
            env = make_env(n, a, dev, **kw)
            env.reset()
            acts = make_actions(8, n, args.actions, dev, seed=50 + cid)
            k = max(50, min(K, int(5e7 // n)))
            k -= k % 50
            sec, group = time_graph(env, acts, k, 24, group=50)
            st = env.episode_stats()
            # algorithmic bytes per env-step of the variant: + the FP64 RunningMeanStd planes (27 doubles read and written),
            # + last_rpm_sum (drag / ground effect), + the [N,4] aux plane of the rewards that keep one (read and written)
            rid = kw.get("reward_id", L.DN_REWARD_DEFAULT)
            bytes_per = (BYTES_PER_ENV_STEP + (2 * 27 * 8 if kw.get("normalize_obs") else 0) + (8 if kw.get("physics") else 0)
                         + (32 if rid in (L.DN_REWARD_REACHING, L.DN_REWARD_BOOTSTRAPPED, L.DN_REWARD_CHAMP) else 0))
            variant = "norm_" if kw.get("normalize_obs") else "phys3_" if kw.get("physics") else f"full_rw{rid}_" if "reward_id" in kw and rid else ""
            kern = "dn::step_kernel<%d,%s,false,%s>" % (3 if kw.get("physics") else 0, "true" if kw.get("normalize_obs") else "false",
                                                        "true" if ("reward_id" in kw and rid) else "false")
            rl = roofline(n, sec / k, substeps=S, bytes_per=bytes_per, variant=variant, kernel=kern)
            rl["l2"] = "fits L2 (graph replay over one handle)" if n * (bytes_per - 112) < 126e6 else "larger than L2"
            out.append({"config": cid, "shape": name, "envs": n, "substeps": S, "value": n * k / sec, "unit": UNIT,
                        "us_per_launch": 1e6 * sec / k, "achieved_gbs": rl["achieved"], "roofline": rl, "steps": k,
                        "episodes_finished": int(st["episodes"]), "timing": "CUDA-graph replay, 50 steps per graph"})
            env.close()
            del env, acts
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            out.append({"config": cid, "shape": name, "error": str(ex)[:200]})
    return out


def make_actions(n_buf, n_envs, mode, device, seed):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    u = torch.rand(n_buf, n_envs, 4, generator=g, device=device) * 2 - 1
    return u.contiguous() if mode == "saturating" else (HOVER + 0.002 * u).contiguous()


def time_flushed(env, acts, K, W, flush_buf):
    """K launches, each bracketed by its own CUDA-event pair on the launching stream, L2 flushed
    (a write larger than L2) between them outside the timed brackets."""
    import torch
    A = acts.shape[0]
    for k in range(W):
        env.step(acts[k % A])
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for k in range(K):
        flush_buf.fill_(k & 1)
        starts[k].record()
        env.step(acts[(W + k) % A])
        ends[k].record()
    torch.cuda.synchronize()
    per = np.array([s.elapsed_time(e) for s, e in zip(starts, ends)])     # ms
    return float(per.sum()) * 1e-3, per


def time_rotating(args, dev, N, K, W, rank, n_handles=None, on_timed=None, want_outputs=False):
    """`inputs larger than L2`: M independent N-env handles (state + actions + outputs of all of them > 126 MB L2) are
    stepped round-robin, one launch per handle, replayed from CUDA graphs on one stream.  The timed region is EXACTLY K
    launches inside one CUDA-event pair.  Right before it the graphs that precede it in the rotation are replayed, untimed:
    that leaves each timed launch's state, actions and output lines in HBM rather than in L2.  How often each handle has
    been stepped depends on the arguments alone, so the outputs of the last timed launch are the same from run to run;
    with `want_outputs` they are returned as numpy arrays (what `env.step` hands its caller)."""
    import torch
    per_handle = N * (BYTES_PER_ENV_STEP - 112)          # state planes once + actions + outputs, bytes resident per handle
    M = n_handles or max(8, int(np.ceil(160e6 / per_handle)))
    if not n_handles and K < M:
        M = K * -(-M // K)                               # whole number of K-launch blocks per rotation
    envs = [make_env(N, args, dev, env_id_offset=rank * N) for _ in range(M)]
    for e in envs:
        e.reset()
    acts = make_actions(M, N, args.actions, dev, seed=4321 + rank)
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for _ in range(max(24, -(-W // M))):             # >= W untimed warm-up steps (whole rotations), >= 24 per handle:
                                                         # episodes are de-phased (steady-state reset mix), as in the sweep
            for m, e in enumerate(envs):
                e.step(acts[m])
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize()
    # graph b holds the K launches of handles (b*K + j) % M, j < K: the graphs continue one rotation, so every launch of
    # the last (timed) graph finds its handle last stepped M launches earlier (> 126 MB ago).  At least two graphs: one
    # graph replayed twice would bring some handles back after fewer than M launches unless M divides K
    n_graphs = max(2, -(-M // K))
    graphs = []
    for b in range(n_graphs):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for j in range(K):
                m = (b * K + j) % M
                envs[m].step(acts[m])
        graphs.append(g)
    if on_timed:
        on_timed(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for g in graphs[:-1]:                                # untimed, not synchronised: the timed replay queues behind them
        g.replay()
    e0.record()
    graphs[-1].replay()
    e1.record()
    torch.cuda.synchronize()
    if on_timed:
        on_timed(False)
    sec = e0.elapsed_time(e1) * 1e-3
    last = None
    if want_outputs:                                     # env.step returns views of these persistent output tensors
        e = envs[(n_graphs * K - 1) % M]
        last = {k: getattr(e, k).cpu().numpy() for k in ("obs", "reward", "done", "found_targets")}
    eps = sum(int(e.episode_stats()["episodes"]) for e in envs[:4])
    for e in envs:
        e.close()
    del envs, acts, graphs
    torch.cuda.empty_cache()
    return sec, K, M, per_handle * M, eps, n_graphs, last


def time_launch_floor(env, K, flush_buf):
    """The same two measurement harnesses around a (near-)empty kernel of the same library -- action_map_kernel over 4
    floats: (a) per-launch CUDA-event brackets with the L2 flush in between, (b) CUDA-graph replay back to back.  What
    is left of a 4096-env step after subtracting these is the step kernel's own time."""
    import torch
    a = torch.zeros(4, dtype=torch.float32, device=env.device)
    for _ in range(10):
        env.action_to_rpm(a)
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for k in range(K):
        flush_buf.fill_(k & 1)
        starts[k].record()
        env.action_to_rpm(a)
        ends[k].record()
    torch.cuda.synchronize()
    bracket = float(np.mean([s.elapsed_time(e) for s, e in zip(starts, ends)])) * 1e3
    s = torch.cuda.Stream(device=env.device)
    s.wait_stream(torch.cuda.current_stream(env.device))
    out = torch.empty_like(a)
    import ctypes as C
    from drl_dronenavigation_b200 import _lib as L

    def tiny():
        L.check(env._lib.dn_action_to_rpm(env._handle, a.data_ptr(), out.data_ptr(), 4,
                                          C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)))
    with torch.cuda.stream(s):
        tiny()
    torch.cuda.current_stream(env.device).wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for _ in range(50):
            tiny()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(max(K // 50, 1)):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return {"event_bracket_us": bracket, "graph_replay_us": e0.elapsed_time(e1) * 1e3 / (max(K // 50, 1) * 50),
            "kernel": "dn::action_map_kernel over 4 floats (empty-kernel stand-in)"}


def time_graph(env, acts, K, W, group=None, min_timed_s=0.02):
    """K launches replayed from CUDA graphs of `group` steps each, back to back, one event pair around all."""
    import torch
    A = acts.shape[0]
    group = group or min(K, A, 50)
    while K % group:
        group -= 1
    s = torch.cuda.Stream(device=env.device)
    s.wait_stream(torch.cuda.current_stream(env.device))
    with torch.cuda.stream(s):
        for k in range(max(W, 3)):
            env.step(acts[k % A])
    torch.cuda.current_stream(env.device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for k in range(group):
            env.step(acts[k % A])
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K // group):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    est = max(e0.elapsed_time(e1) * 1e-3, 1e-6)
    R = int(max(1, min(100000, np.ceil(min_timed_s / est))))   # K launches repeated R times inside one event pair
    e0.record()
    for _ in range(R * (K // group)):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / R, group


def time_plain(env, acts, K, W):
    """K plain launches back to back (no graph), one event pair around all."""
    import torch
    A = acts.shape[0]
    for k in range(W):
        env.step(acts[k % A])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        env.step(acts[(W + k) % A])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(n_envs, substeps, variant=""):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of step_kernel from the committed `ncu --set full`
    capture of the same configuration (profiles/ncu_summary_r*.json, written by tools/summarize_profiles*.py from the
    reports; `variant` = the capture's prefix: "" plain, "norm_", "phys3_", "full_rw<id>_"); the latest round that
    holds the capture wins; None if that configuration was not captured."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_summary_r*.json"))):
        try:
            with open(path) as f:
                d = json.load(f)
            rec = d.get(f"{variant}n{n_envs}_s{substeps}") or (d.get(f"prof_n{n_envs}_s{substeps}.ncu-rep") if not variant else None)
            if rec and "traffic_bytes" in rec:
                best = float(rec["traffic_bytes"])
        except Exception:  # noqa: BLE001
            pass
    return best


def roofline(n_envs, sec_per_launch, traffic=None, substeps=None, bytes_per=BYTES_PER_ENV_STEP, variant="", kernel="dn::step_kernel<0,false,false,false>"):
    peak, src = peaks()
    if traffic is None and substeps is not None:
        traffic = ncu_traffic(n_envs, substeps, variant)
    achieved = bytes_per * n_envs / sec_per_launch / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "kernel": kernel, "bytes_per_env_step": bytes_per, "envs_per_launch": n_envs,
            "algorithmic_bytes_per_launch": bytes_per * n_envs, "us_per_launch": sec_per_launch * 1e6, "peak_source": src}


def run_sac(args, dev, world, rank, barrier, max_over_ranks):
    """SAC samples/s end to end on BASELINE configs[3]: 16384 envs per GPU, circle track, drag + ground-effect physics,
    reference SAC-branch hyper-parameters (train_freq 3 env steps, 5 gradient steps of batch 1024, twin critics
    [256,256,128], actor [256,256]); two flat-bucket NCCL all-reduces per gradient step under torchrun."""
    import copy
    import torch
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.sac import SACConfig, SACTrainer
    a = copy.copy(args)
    a.track = "circle"
    n = args.sac_envs
    env = make_env(n, a, dev, env_id_offset=rank * n, physics=Physics.PYB_GND_DRAG_DW, normalize_obs=not args.no_norm_obs)
    tr = SACTrainer(env, SACConfig(learning_starts=2 * 3 * n * world))     # two collection-only iterations, then updates
    for _ in range(4):
        tr.train_iteration()                                               # warm-up (past learning_starts)
    barrier()
    l0 = env.launch_count
    t0 = time.perf_counter()
    outs = [tr.train_iteration() for _ in range(args.sac_iters)]
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    barrier()
    samples = sum(o["samples"] for o in outs)
    res = {"value": samples / dt, "unit": "samples/s (env-steps/s incl. actor inference and SAC updates)", "envs_per_gpu": n,
           "iterations": args.sac_iters, "train_freq": tr.cfg.train_freq, "gradient_steps": tr.cfg.gradient_steps,
           "batch_size": tr.cfg.batch_size, "gradient_steps_run": sum(o["gradient_steps"] for o in outs),
           "physics": "DYN + drag + ground effect", "track": "circle", "substeps": args.substeps,
           "critic_loss": outs[-1].get("critic_loss"), "ent_coef": outs[-1].get("ent_coef"),
           "allreduce_calls": tr.learner.g_critic.calls + tr.learner.g_actor.calls, "gpu_launches": int(env.launch_count - l0),
           "replay_transitions": len(tr.buffer)}
    env.close()
    return res


def run_ppo(args, dev, world, rank, barrier, max_over_ranks):
    """PPO samples/s end to end on `--ppo-envs` envs per GPU: rollout (policy inference + fused env step, all on
    device) + GAE kernel + the PPO update (10 epochs, clipped losses, KL early stop) with ONE flat-gradient
    NCCL all-reduce per optimiser step.  Reference hyper-parameters; rollout length and minibatch scaled."""
    import torch
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    import copy
    a = copy.copy(args)
    a.track = args.ppo_track
    # the reference's wrapper stack: every env is wrapped in NormalizeObservation (PBDroneSimulator.py:181) -> the NORM kernel variant
    env = make_env(args.ppo_envs, a, dev, env_id_offset=rank * args.ppo_envs, normalize_obs=not args.no_norm_obs)
    T = args.ppo_rollout
    cfg = PPOConfig(n_steps=T, batch_size=max(512, (T * args.ppo_envs) // 32), update_impl=args.ppo_impl, mlp_precision=args.ppo_precision)
    tr = PPOTrainer(env, cfg, rollout_steps=T)
    for _ in range(2):
        tr.train_iteration()                               # warm-up (kernel loading, plans, graph capture, allocator)
    barrier()
    l0 = env.launch_count
    t0 = time.perf_counter()
    outs = [tr.train_iteration() for _ in range(args.ppo_iters)]
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    barrier()
    samples = world * args.ppo_envs * T * args.ppo_iters
    res = {"value": samples / dt, "unit": "samples/s (env-steps/s incl. policy inference and PPO update)",
           "envs_per_gpu": args.ppo_envs, "rollout_steps": T, "iterations": args.ppo_iters, "track": a.track, "substeps": args.substeps,
           "minibatch": cfg.batch_size, "epochs_run": [o["epochs"] for o in outs], "minibatches_run": [o["minibatches"] for o in outs],
           "rollout_s": sum(o["rollout_s"] for o in outs), "update_s": sum(o["update_s"] for o in outs),
           "rollout_s_each": [round(o["rollout_s"], 5) for o in outs], "update_s_each": [round(o["update_s"], 5) for o in outs],
           "env_share_of_rollout": None, "allreduce_calls": tr.learner.allreduce_calls, "allreduce_bytes": tr.learner.n_params * 4, "allreduce_impl": getattr(tr.learner, "allreduce_impl", "nccl" if world > 1 else "none"),
           "gpu_launches": int(env.launch_count - l0), "approx_kl": outs[-1]["approx_kl"],
           "normalize_obs": not args.no_norm_obs, "update_impl": outs[-1].get("impl", "torch/" + cfg.matmul_precision),
           "optimizer_steps": [o.get("optimizer_steps") for o in outs], "update_us_per_minibatch": 1e6 * sum(o["update_s"] for o in outs) / max(1, sum(o["minibatches"] for o in outs)),
           "policy": "2 x MLP 13-512-512-256 (pi, vf), Tanh; update + rollout forward: hand-written sm_100a kernels (tcgen05 BF16 hi/lo planes, "
                     "FP32 TMEM accumulation) unless update_impl says torch"}
    impl_ar = res["allreduce_impl"]
    res["collective"] = ("none (1 GPU)" if world == 1 else
                         "sum of one flat FP32 gradient bucket per optimiser step over NVLink peer memory (the library's own kernel, inside the minibatch graph)"
                         if impl_ar == "peer" else "NCCL all-reduce of one flat FP32 gradient bucket per optimiser step")
    # aggregate tensor-core roofline of the update: forward + dgrad + wgrad of both MLPs = (2 + 2 + 2) x sum(in x out) flop per sample and net,
    # times the BF16 products issued per FP32 product (3 in the FP32-faithful mode), over the WHOLE update time (gather, heads, losses,
    # reductions, clip and Adam included), against the measured dense BF16 rate
    try:
        arch = tuple(cfg.pi_arch)
        dims = [(64, arch[0])] + [(arch[i], arch[i + 1]) for i in range(len(arch) - 1)]          # the 13-dim observation is padded to K = 64
        passes = 3 if "bf16x3" in res["update_impl"] else 1
        flop_per_sample = 2 * (4 * sum(i * o for i, o in dims) + 2 * sum(i * o for i, o in dims[1:])) * passes   # no dgrad below the first layer
        n_samples = sum(o["minibatches"] for o in outs) * cfg.batch_size
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak_tf = float(json.load(f)["bf16_tflops"])
        ach = flop_per_sample * n_samples / max(res["update_s"], 1e-9) / 1e12
        if "fused" in res["update_impl"]:
            res["roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": None,
                               "kernel": "dnmma::umma_gemm<KIND, 256, 2> (all contractions of the update; per-kernel table: profiles/ppo_r02.md)",
                               "flop_counting": f"{passes} BF16 product(s) per FP32 product; whole update time incl. gather, heads, reductions, clip, Adam",
                               "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops)"}
    except Exception:  # noqa: BLE001
        pass
    env.close()
    return res


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from drl_dronenavigation_b200 import _lib
    _lib.lib()             # the library build() left in the tree: nothing is compiled here, nothing is written there
    K, W = args.steps, max(args.warmup, 3)
    N = args.envs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    env = make_env(N, args, dev, env_id_offset=rank * N)
    env.reset()
    A = max(8, min(1000, (64 << 20) // (N * 16)))
    acts = make_actions(A, N, args.actions, dev, seed=1234 + rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)

    # ---- headline: EXACTLY K launches on inputs larger than L2 (rotating handles), one event pair -------------
    # (timing rule: "flush L2 between timed iterations OR use inputs larger than L2" -- this is the second form; the
    #  first form is reported below as `flushed_event_bracket`, where two event records per launch cost ~6 us of
    #  harness time against a ~3 us kernel, see `launch_floor`)
    barrier()
    win = {}
    def around_timed(start):          # barrier + synchronize on both sides of the timed region, on every rank
        barrier()
        win["t0" if start else "t1"] = time.time()
    sec, k_r, m_r, bytes_r, eps_r, n_graphs, last = time_rotating(args, dev, N, K, W, rank, n_handles=args.rotating_handles,
                                                                  on_timed=around_timed, want_outputs=bool(args.dump_outputs))
    assert k_r == K
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    barrier()
    sec = max_over_ranks(sec)
    value = world * N * K / sec
    l2_note = ("PROFILING RUN with a reduced number of handles (L2-resident): " if args.rotating_handles else "") + \
              (f"inputs larger than L2: {m_r} independent {N}-env handles = {bytes_r / 1e6:.0f} MB of state + actions + outputs "
               "(> 126 MB L2) stepped round-robin from CUDA graphs on one stream, so every launch reads its inputs from HBM; "
               "no flush kernel, one CUDA-event pair around the K launches")

    # ---- the other sanctioned form: L2 flushed between launches, per-launch CUDA-event brackets ----------------
    barrier()
    sec_f, per = time_flushed(env, acts, K, W, flush)
    barrier()
    sec_f = max_over_ranks(sec_f)
    clocks = sampler.stop(win.get("t0", time.time() - 1), max(win.get("t1", time.time()), win.get("t0", 0) + 0.05))
    flushed = {"value": world * N * K / sec_f, "unit": UNIT, "us_per_launch": 1e6 * sec_f / K,
               "l2": "flushed between timed launches (256 MiB fill, outside the per-launch event brackets)"}

    # ---- same workload, L2-resident, CUDA-graph replay (launch-latency regime) -------------------
    barrier()
    sec_g, group = time_graph(env, acts, K, W)
    sec_g = max_over_ranks(sec_g)
    barrier()
    sec_p = max_over_ranks(time_plain(env, acts, K, W))
    resident = {"value": world * N * K / sec_g, "unit": UNIT, "us_per_launch": 1e6 * sec_g / K, "cuda_graph_steps": group,
                "plain_launch_value": world * N * K / sec_p, "plain_us_per_launch": 1e6 * sec_p / K,
                "note": "state (0.9 MB) stays in L2 between launches, as in real use at this batch size"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * sec / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": bench_config(args, world),
            "timed_region_s": sec,
            "timing": {"l2": l2_note, "handles": m_r, "graphs": n_graphs, "launches_per_graph": K,
                       "timed_region_s": sec, "launches_in_timed_region": K,
                       "note": "ms_per_step = timed_region_s / steps: exactly `steps` launches (one graph replay) inside ONE "
                               "CUDA-event pair; the graphs before it in the rotation are replayed right before it"},
            "physics_steps_per_s": value * args.substeps,
            "clocks": clocks, "gpu_launches": K, "l2_resident": resident, "flushed_event_bracket": flushed,
            "episodes_finished_sample": eps_r}

    # ---- single-GPU extras on rank 0 only: roofline, sweep, e2e, cpu baseline --------------------
    if world == 1:
        line["roofline"] = roofline(N, sec / K, substeps=args.substeps)
        line["roofline"]["note"] = "launch/latency-bound at this batch size: 1.2 MB per launch is ~0.2 us of HBM time"
        try:
            line["launch_floor"] = time_launch_floor(env, min(K, 300), flush)
        except Exception as ex:  # noqa: BLE001
            line["launch_floor"] = {"error": str(ex)[:200]}
        sweep = []
        for n_big in args.sweep:
            try:
                e2 = make_env(n_big, args, dev)
                e2.reset()
                a2 = make_actions(4, n_big, args.actions, dev, seed=99)
                k2 = max(10, min(K, int(2e8 // n_big)))
                s2 = time_plain(e2, a2, k2, 24)      # 24 warm-up steps: episodes are de-phased (steady-state reset mix)
                rf = roofline(n_big, s2 / k2, substeps=args.substeps)
                sweep.append({"envs": n_big, "value": n_big * k2 / s2, "us_per_launch": 1e6 * s2 / k2, "steps": k2,
                              "roofline_frac": rf["frac"], "achieved_gbs": rf["achieved"],
                              "working_set_mb": n_big * (BYTES_PER_ENV_STEP - 16) / 1e6, "l2": "inputs larger than L2" if n_big * 224 > 126e6 else "fits L2"})
                if n_big == max(args.sweep):
                    line["roofline_hbm"] = rf
                e2.close()
                del e2, a2
                torch.cuda.empty_cache()
            except Exception as ex:  # noqa: BLE001
                sweep.append({"envs": n_big, "error": str(ex)[:200]})
        line["sweep"] = sweep
        if not args.no_configs:
            line["baseline_configs"] = baseline_configs(args, dev, K)
        # S = 1 variant of the largest batch (reference default 240/240 Hz): HBM-bound regime
        try:
            import copy
            a1 = copy.copy(args); a1.substeps = 1
            n_big = max(args.sweep)
            e3 = make_env(n_big, a1, dev); e3.reset()
            a3 = make_actions(4, n_big, args.actions, dev, seed=98)
            k3 = max(10, min(K, int(2e8 // n_big)))
            s3 = time_plain(e3, a3, k3, 24)
            line["roofline_hbm_s1"] = roofline(n_big, s3 / k3, substeps=1)
            line["roofline_hbm_s1"]["substeps"] = 1
            e3.close(); del e3, a3
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            line["roofline_hbm_s1"] = {"error": str(ex)[:200]}

    # ---- e2e: C-ABI host-buffer call, pinned host actions -> H2D -> kernel -> D2H results ---------
    # Headline form: the handle's own pinned slab (dn_host_buffers): per step the caller writes that step's actions into the
    # pinned slab, dn_step_host replays one captured graph (H2D DMA of the actions, fused kernel, D2H DMA of the packed
    # results) and returns when the results are in the slab.  K steps form a block; blocks are repeated until the timed
    # region is >= 50 ms (wall clock needs it), the mean block is reported.
    D = env.obs_dim
    h_act = torch.empty(A, N, 4, dtype=torch.float32).pin_memory()
    h_act.copy_(acts.cpu())
    a_np = h_act.numpy()
    torch.cuda.synchronize()
    slab_io, slab = env.host_buffers(with_episode_info=False)

    def e2e_block(step_fn, n_steps, k0):
        t0 = time.perf_counter()
        for k in range(n_steps):
            step_fn((k0 + k) % A)
        return time.perf_counter() - t0

    def e2e_measure(step_fn):
        for k in range(W):
            step_fn(k % A)
        est = max(e2e_block(step_fn, K, W), 1e-6)
        R = int(max(1, min(100000, np.ceil(0.05 / est))))
        barrier()
        l0 = env.launch_count
        tot = 0.0
        for r in range(R):
            tot += e2e_block(step_fn, K, W + r * K)
        launches_ = env.launch_count - l0
        barrier()
        return max_over_ranks(tot / R), R, launches_

    def step_slab(k):
        np.copyto(slab["actions"], a_np[k])
        env.step_host(slab_io)
    e2e_sec, e2e_reps, e2e_launches = e2e_measure(step_slab)
    checksum = float(slab["reward"][:8].sum())           # the results are read on the host
    e2e_slab = {"value": world * N * K / e2e_sec, "unit": UNIT, "h2d_bytes_per_step": N * 16,
                   "d2h_bytes_per_step": N * (D * 4 + 4 + 1 + 4), "us_per_step": 1e6 * e2e_sec / K, "reps": e2e_reps,
                   "api": "dn_host_buffers + dn_step_host (C ABI): the step's actions are written into the handle's pinned host slab, one "
                          "captured graph per step = H2D DMA (actions) -> fused kernel -> D2H DMA (obs, reward, found_targets, done, "
                          "completion word); the host polls the completion word",
                   "gpu_launches": int(e2e_launches), "reward_checksum": checksum}
    # the previous form, kept as a comparison line: caller-owned pinned buffers, the kernel reads / writes them over PCIe itself
    h_obs = torch.empty(N, D, dtype=torch.float32).pin_memory()
    h_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    h_done = torch.empty(N, dtype=torch.uint8).pin_memory()
    h_found = torch.empty(N, dtype=torch.int32).pin_memory()
    ios = [env._make_io(h_act[k], h_obs, h_rew, h_done, None, h_found) for k in range(A)]
    zc_sec, zc_reps, zc_launches = e2e_measure(lambda k: env.step_host(ios[k]))
    e2e_zc = {"value": world * N * K / zc_sec, "unit": UNIT, "h2d_bytes_per_step": N * 16, "d2h_bytes_per_step": N * (D * 4 + 4 + 1 + 4),
              "us_per_step": 1e6 * zc_sec / K, "reps": zc_reps, "gpu_launches": int(zc_launches), "reward_checksum": float(h_rew[:8].sum()),
              "api": "dn_step_host (C ABI) with caller-owned pinned host buffers, zero copy: the fused kernel reads that step's actions from and "
                     "writes obs, reward, found_targets, done to host memory over PCIe (64 KiB in, 244 KiB out per step); its last CTA "
                     "writes a completion word the host polls -- one launch per step, no DMA engine, no stream query"}
    # third form: the same call and the same caller-owned pinned buffers with the resident step server on (dn_host_server): the
    # step kernel stays on the GPU between calls, the host rings a doorbell word per step instead of launching
    forms = {"zero_copy": e2e_zc, "slab_graph": e2e_slab}
    try:
        env.host_server(args.server_idle_us)
        s0 = env.host_server_stats()
        srv_sec, srv_reps, srv_launches = e2e_measure(lambda k: env.step_host(ios[k]))
        s1 = env.host_server_stats()
        env.host_server(0)
        forms["server"] = {"value": world * N * K / srv_sec, "unit": UNIT, "h2d_bytes_per_step": N * 16, "d2h_bytes_per_step": N * (D * 4 + 4 + 1 + 4),
                           "us_per_step": 1e6 * srv_sec / K, "reps": srv_reps, "gpu_launches": int(srv_launches),
                           "server_steps": s1["steps"] - s0["steps"], "server_residencies": s1["residencies"] - s0["residencies"],
                           "server_idle_us": args.server_idle_us, "reward_checksum": float(h_rew[:8].sum()),
                           "api": "dn_host_server + dn_step_host (C ABI) with caller-owned pinned host buffers: the step kernel (dn_step_many "
                                  "variant) is RESIDENT; per step the host writes that step's actions, rings a doorbell word in pinned memory "
                                  "and polls the completion word; the kernel reads the actions from and writes obs, reward, found_targets, "
                                  "done to host memory over PCIe (64 KiB in, 244 KiB out per step) -- no launch per step"}
    except Exception as ex:  # noqa: BLE001
        forms["server"] = {"error": str(ex)[:200], "value": 0.0}
    # all forms move the same bytes between host and device inside the timed region; the headline is the fastest one at this batch size
    order = sorted(forms, key=lambda k: -forms[k]["value"])
    line["e2e"] = dict(forms[order[0]], form=order[0])
    line["e2e_alternative"] = dict(forms[order[1]], form=order[1])
    line["e2e_forms"] = {k: {kk: v.get(kk) for kk in ("value", "us_per_step", "gpu_launches", "error") if kk in v} for k, v in forms.items()}
    if world == 1:
        # the staged variant of the same call (pageable numpy buffers: H2D copy -> kernel -> D2H copies)
        p_act = h_act.numpy().copy()
        p_obs, p_rew = np.empty((N, D), np.float32), np.empty(N, np.float32)
        p_done, p_found = np.empty(N, np.uint8), np.empty(N, np.int32)
        from drl_dronenavigation_b200 import _lib as L
        pios = []
        for k in range(A):
            io = L.dn_step_io()
            io.actions, io.obs, io.reward, io.done, io.found_targets = (p_act[k].ctypes.data, p_obs.ctypes.data, p_rew.ctypes.data,
                                                                        p_done.ctypes.data, p_found.ctypes.data)
            pios.append(io)
        ks = min(K, 300)
        for k in range(5):
            env.step_host(pios[k % A])
        t0 = time.perf_counter()
        for k in range(ks):
            env.step_host(pios[k % A])
        dts = time.perf_counter() - t0
        line["e2e_staged"] = {"value": N * ks / dts, "unit": UNIT, "us_per_step": 1e6 * dts / ks,
                              "api": "dn_step_host with pageable host buffers (staged H2D / D2H copies)"}
    if world == 1 and not args.no_vecenv:
        # the SB3 VecEnv protocol on top of the same call (numpy in / numpy out + per-env info dicts)
        from drl_dronenavigation_b200.vec_env import GpuDroneVecEnv
        targets, init, dim, is_circle = track_setup(args.track)
        venv = GpuDroneVecEnv(N, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=240 // args.substeps,
                              circle=is_circle, include_distance=True, normalize_actions=True, normalize_obs=True, device=dev)
        venv.reset()
        a_np = h_act.numpy()
        kv = min(K, 200)
        for k in range(3):
            venv.step(a_np[k % A])
        t0 = time.perf_counter()
        for k in range(kv):
            venv.step(a_np[k % A])
        dtv = time.perf_counter() - t0
        line["e2e_vecenv"] = {"value": N * kv / dtv, "unit": UNIT, "us_per_step": 1e6 * dtv / kv,
                              "api": "GpuDroneVecEnv.step (SB3 VecEnv protocol incl. NormalizeObservation, Monitor, info dicts)"}
        venv.close()
        # BASELINE configs[0], the reference's own CPU-runnable case: num_envs = 12, 240/240 Hz, circle track, per-env
        # NormalizeObservation + Monitor, through the same SB3 VecEnv protocol the reference's SubprocVecEnv speaks
        try:
            import copy
            a0 = copy.copy(args); a0.substeps, a0.track = 1, "circle"
            t12, i12, d12, c12 = track_setup("circle")
            a12 = (np.random.default_rng(0).uniform(-1, 1, size=(64, 12, 4))).astype(np.float32)
            k12, us12 = 3000, {}
            for path in ("zero_copy", "server"):
                v12 = GpuDroneVecEnv(12, t12, aviary_dim=d12, initial_xyzs=i12, pyb_freq=240, ctrl_freq=240, circle=c12,
                                     include_distance=True, normalize_actions=True, normalize_obs=True, device=dev, host_path=path)
                v12.reset()
                for k in range(200):
                    v12.step(a12[k % 64])
                t0 = time.perf_counter()
                for k in range(k12):
                    v12.step(a12[k % 64])
                us12[path] = 1e6 * (time.perf_counter() - t0) / k12
                v12.close()
            best12 = min(us12, key=us12.get)
            line["e2e_vecenv_config1"] = {"value": 12 * 1e6 / us12[best12], "unit": UNIT, "us_per_step": us12[best12], "num_envs": 12,
                                          "substeps": 1, "host_path": best12, "us_per_step_by_host_path": us12,
                                          "api": "GpuDroneVecEnv.step, README configuration (12 envs, 240/240 Hz)",
                                          "note": "the reference's 4 h / 1e7 steps anecdote corresponds to ~700 env-steps/s end to end incl. PPO"}
        except Exception as ex:  # noqa: BLE001
            line["e2e_vecenv_config1"] = {"error": str(ex)[:200]}

    # ---- PPO SPS end to end (BASELINE configs[2]): device-resident rollout + update, NCCL gradient all-reduce ----
    if not args.no_ppo:
        try:
            line["ppo"] = run_ppo(args, dev, world, rank, barrier, max_over_ranks)
        except Exception as ex:  # noqa: BLE001
            line["ppo"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}

    if not args.no_ppo:
        try:
            line["sac"] = run_sac(args, dev, world, rank, barrier, max_over_ranks)
        except Exception as ex:  # noqa: BLE001
            line["sac"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}

    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(args.track, args.substeps, budget_s=args.cpu_budget)
        line["pybullet_cpu"] = pybullet_cpu()
        try:
            line["cpu_baseline_batched"] = cpu_baseline_batched(args.track, args.substeps, args.envs)
        except Exception as ex:  # noqa: BLE001
            line["cpu_baseline_batched"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
    elif world > 1:
        line["cpu_baseline"] = None
    env.close()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True      # the tree may be read-only: the modules imported from it leave no __pycache__ there
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU (BASELINE configs[1]: 4096)")
    ap.add_argument("--substeps", type=int, default=8, help="pyb_freq / ctrl_freq (240/30 Hz -> 8)")
    ap.add_argument("--track", default="circle", choices=["circle", "reaching"])
    ap.add_argument("--actions", default="saturating", choices=["saturating", "hover_band"])
    ap.add_argument("--sweep", type=int, nargs="*", default=[65536, 1 << 20, 1 << 22])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ppo", action="store_true")
    ap.add_argument("--ppo-envs", type=int, default=65536, help="BASELINE configs[2]: 65536 envs per GPU")
    ap.add_argument("--ppo-rollout", type=int, default=16)
    ap.add_argument("--ppo-iters", type=int, default=2)
    ap.add_argument("--ppo-track", default="reaching", choices=["circle", "reaching"])
    ap.add_argument("--sac-envs", type=int, default=16384, help="BASELINE configs[3]: 16384 envs")
    ap.add_argument("--sac-iters", type=int, default=20)
    ap.add_argument("--no-vecenv", action="store_true")
    ap.add_argument("--no-norm-obs", dest="no_norm_obs", action="store_true",
                    help="learner lines on raw observations (labelled deviation; the reference always normalises, PBDroneSimulator.py:181)")
    ap.add_argument("--ppo-precision", default="bf16x3", choices=["bf16x3", "bf16"], help="arithmetic of the fused PPO update's contractions")
    ap.add_argument("--ppo-impl", default="auto", choices=["auto", "fused", "torch"])
    ap.add_argument("--server-idle-us", type=int, default=2000,
                    help="idle time after which the resident step server of the e2e 'server' form leaves the GPU")
    ap.add_argument("--rotating-handles", type=int, default=None,
                    help="override the number of rotating handles of the headline measurement (default: enough for > 126 MB; "
                         "the ncu launch-list pass uses a small number so that the capture window covers the timed region)")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-BASELINE-config step-only lines")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write obs, reward, done and found_targets of the last timed step (the handle it stepped) as DIR/<name>.npy; "
                         "the inputs depend on the arguments only, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs: only the GPU arm (--impl b200) writes its outputs")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
