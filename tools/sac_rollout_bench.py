"""SAC collection and whole SAC iterations, rollout_impl "torch" against "fused" (dn_sac_act + each collection phase replayed
from a CUDA graph), at BASELINE config 4 (16 384 envs, circle track, drag + ground effect, NormalizeObservation) and at 4096 envs.

    python tools/sac_rollout_bench.py [--rounds 20] [--warmup 4] [--envs 16384,4096] [--out FILE]

Per env count both trainers are built with the reference SAC hyper-parameters (train_freq 3, 5 gradient steps of batch 1024) and
learning_starts = two collection phases, warmed up with `--warmup` iterations (past learning_starts; the fused trainer captures
its collection graph at the second phase after it), then timed in alternation, A B A B ..., `--rounds` iterations each.
collect_s is SACTrainer.train_iteration's device-event time of the collection phase; iteration_s its host clock around the
whole iteration, which ends in a device synchronise.  Prints one JSON line per env count and implementation, with the card's
name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.rollout_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--envs", type=str, default="16384,4096")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    import torch
    import bench
    from drl_dronenavigation_b200 import Physics
    from drl_dronenavigation_b200.batched_env import BatchedDroneEnv
    from drl_dronenavigation_b200.sac import SACConfig, SACTrainer
    if not torch.cuda.is_available():
        raise SystemExit("sac_rollout_bench.py needs a CUDA device")
    name, power = card()
    targets, init, dim, is_circle = bench.track_setup("circle")
    lines = []
    for N in (int(v) for v in args.envs.split(",")):
        trainers = {}
        for impl in ("torch", "fused"):
            env = BatchedDroneEnv(N, targets, threshold=0.3, discount=0.999, max_steps=4096, aviary_dim=dim, initial_xyzs=init, pyb_freq=240,
                                  ctrl_freq=30, cylinder=True, circle=is_circle, include_distance=True, normalize_actions=True,
                                  normalize_obs=True, physics=Physics.PYB_GND_DRAG_DW, device="cuda:0")
            trainers[impl] = SACTrainer(env, SACConfig(learning_starts=2 * 3 * N, rollout_impl=impl))
        for tr in trainers.values():
            for _ in range(args.warmup):
                tr.train_iteration()
        times = {impl: {"collect_s": [], "iteration_s": []} for impl in trainers}
        for _ in range(args.rounds):
            for impl, tr in trainers.items():
                o = tr.train_iteration()
                times[impl]["collect_s"].append(o["collect_s"])
                times[impl]["iteration_s"].append(o["seconds"])
        for impl, tr in trainers.items():
            t = times[impl]
            med = {k: statistics.median(v) for k, v in t.items()}
            line = {"envs": N, "train_freq": tr.cfg.train_freq, "gradient_steps": tr.cfg.gradient_steps, "batch_size": tr.cfg.batch_size,
                    "samples_per_iteration": tr.cfg.train_freq * N, "rollout_impl": impl,
                    "collect_s_median": med["collect_s"], "iteration_s_median": med["iteration_s"],
                    "collect_share": med["collect_s"] / med["iteration_s"], "samples_per_s": tr.cfg.train_freq * N / med["iteration_s"],
                    "collect_s": t["collect_s"], "iteration_s": t["iteration_s"], "rounds": args.rounds, "warmup": args.warmup,
                    "graph": impl == "fused" and tr._collect_graph is not None, "gpu": name, "power_limit": power,
                    "physics": "DYN + drag + ground effect", "normalize_obs": True,
                    "timing": "collect_s: CUDA events around the collection phase; iteration_s: host clock ending in a device "
                              "synchronise; A/B alternated"}
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
