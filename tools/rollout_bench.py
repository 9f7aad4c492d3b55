"""Rollout collection and whole PPO iterations, rollout_impl "torch" against "fused" (dn_ppo_act + the rollout replayed from a
CUDA graph), on the circle track with NormalizeObservation on.

    python tools/rollout_bench.py [--rounds 5] [--warmup 3] [--shapes 8192x128x16384,65536x16x32768] [--out FILE]

Each shape is envs x rollout steps x minibatch; the minibatch defaults are the README training command's (8192 envs) and the
bench PPO line's (65 536 envs).  Per shape both trainers are built, warmed up with `--warmup` iterations (the fused one captures
its rollout graph at the second), then timed in alternation, A B A B ..., `--rounds` iterations each.  A timing is a host clock
around work that ends in a device synchronise: PPOTrainer.train_iteration's rollout_s (collect_rollouts, including the
bootstrap and GAE) and update_s.  Prints one JSON line per shape and implementation, with the card's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", type=str, default="8192x128x16384,65536x16x32768")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    import torch
    import bench
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench.py needs a CUDA device")
    name, power = card()
    targets, init, dim, is_circle = bench.track_setup("circle")
    lines = []
    for shape in args.shapes.split(","):
        N, T, mb = (int(v) for v in shape.split("x"))
        trainers = {}
        for impl in ("torch", "fused"):
            env = BatchedDroneEnv(N, targets, aviary_dim=dim, initial_xyzs=init, pyb_freq=240, ctrl_freq=30, circle=is_circle,
                                  include_distance=True, normalize_actions=True, normalize_obs=True, device="cuda:0")
            trainers[impl] = PPOTrainer(env, PPOConfig(n_steps=T, batch_size=mb, rollout_impl=impl), rollout_steps=T)
        for impl, tr in trainers.items():
            for _ in range(args.warmup):
                tr.train_iteration()
        times = {impl: {"rollout_s": [], "update_s": [], "iteration_s": []} for impl in trainers}
        for _ in range(args.rounds):
            for impl, tr in trainers.items():
                o = tr.train_iteration()
                times[impl]["rollout_s"].append(o["rollout_s"])
                times[impl]["update_s"].append(o["update_s"])
                times[impl]["iteration_s"].append(o["rollout_s"] + o["update_s"])
        for impl, tr in trainers.items():
            t = times[impl]
            med = {k: statistics.median(v) for k, v in t.items()}
            line = {"shape": {"envs": N, "rollout_steps": T, "minibatch": mb, "samples": N * T}, "rollout_impl": impl,
                    "update_impl": "fused" if tr.learner.fused is not None else "torch",
                    "rollout_s_median": med["rollout_s"], "update_s_median": med["update_s"], "iteration_s_median": med["iteration_s"],
                    "rollout_share": med["rollout_s"] / med["iteration_s"], "rollout_us_per_step": 1e6 * med["rollout_s"] / T,
                    "rollout_s": t["rollout_s"], "update_s": t["update_s"], "rounds": args.rounds, "warmup": args.warmup,
                    "graph": impl == "fused" and tr._rollout_graph is not None, "gpu": name, "power_limit": power,
                    "timing": "host clock around work ending in torch.cuda.synchronize; A/B alternated"}
            print(json.dumps(line), flush=True)
            lines.append(line)
            tr.env.close()
        del trainers
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
