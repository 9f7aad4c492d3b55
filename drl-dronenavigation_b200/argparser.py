"""Command-line flags of the reference (Sol/Utilities/ArgParser.py:6-71) with the defaults of
Sol/Model/parameter_directory/parameter_manager.py:20-38, so existing command lines keep working."""
import argparse
import os

gen_params = {"seed": 1, "num_envs": 12, "learning_rate": 3e-4, "total_timesteps": 10e6, "max_env_steps": 4096,
              "discount": 0.99, "threshold": 0.3, "batch_size": 128, "num_steps": 2048}
def_ppo_params = {"clip_range": 0.1, "ent_coef": 0.2}


def _bool(x):
    x = str(x).lower()
    if x in ("y", "yes", "t", "true", "on", "1"):
        return True
    if x in ("n", "no", "f", "false", "off", "0"):
        return False
    raise ValueError(f"invalid truth value {x!r}")


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser()
    p.add_argument("--exp-name", type=str, default=os.path.basename(__file__).rstrip(".py"))
    p.add_argument("--gym_id", type=str, default="PBDroneEnv")
    p.add_argument("--lib", type=str, default="sb3", choices=["sb3", "ray", "tfa", "clrl"])
    p.add_argument("--run_type", type=str, default="full", choices=["full", "cont", "test", "saved", "learning"])
    p.add_argument("--device", type=str, default="cuda", choices=["cuda", "cpu"])
    p.add_argument("--seed", "-s", type=int, default=gen_params["seed"])
    p.add_argument("--gui", default=False, type=_bool)
    p.add_argument("--obs", type=str, default="pos", choices=["pos", "pos_ext", "rgb"])
    p.add_argument("--profile", default=False, type=_bool)
    p.add_argument("--savemodel", default=True, type=_bool)
    p.add_argument("--vec_check_nan", default=False, type=_bool)
    p.add_argument("--norm_rew", default=False, type=_bool)
    p.add_argument("--clip_rew", default=False, type=_bool)
    p.add_argument("--vec_normalize", default=False, type=_bool)
    p.add_argument("--agent", type=str, default="PPO", choices=["PPO", "SAC", "DDPG", "RECPPO"])
    p.add_argument("--agent-config", type=str, default="default")
    p.add_argument("--num_envs", type=int, default=gen_params["num_envs"])
    p.add_argument("--total_timesteps", type=str, default=gen_params["total_timesteps"])
    p.add_argument("--max_env_steps", type=int, default=gen_params["max_env_steps"])
    p.add_argument("--learning_rate", type=str, default=gen_params["learning_rate"])
    p.add_argument("--discount", type=int, default=gen_params["discount"])
    p.add_argument("--threshold", type=int, default=gen_params["threshold"])
    p.add_argument("--batch_size", type=int, default=gen_params["batch_size"])
    p.add_argument("--num_steps", type=int, default=gen_params["num_steps"])
    p.add_argument("--clip_range", type=int, default=def_ppo_params["clip_range"])
    p.add_argument("--ent_coef", type=int, default=def_ppo_params["ent_coef"])
    p.add_argument("--optimizer", type=str, default="default")
    p.add_argument("--optimizer-config", type=str, default="default")
    p.add_argument("--wandb", type=_bool, default=False, nargs="?", const=True)   # reference default True; no network here
    p.add_argument("--wandb-entity", type=str, default=None)
    p.add_argument("--wandb_rootlog", type=str, default="/wandb")
    p.add_argument("--capture-video", type=_bool, default=False, nargs="?", const=True)
    # additions of this implementation
    p.add_argument("--no_norm_obs", default=False, type=_bool, nargs="?", const=True,
                   help="labelled deviation: train / evaluate on raw observations.  The reference always wraps every env in "
                        "NormalizeObservation (PBDroneSimulator.py:181), which is the default here too (fused, per-env FP64 statistics)")
    p.add_argument("--pyb_freq", type=int, default=240)
    p.add_argument("--ctrl_freq", type=int, default=240)
    p.add_argument("--reward_id", type=int, default=0, help="DN_REWARD_* (include/dronenav.h): 0 PBDroneEnv, 1 dummy_env, "
                   "2 ThrustEnv, 3 HER, 4 reaching-progress (2310.10943), 5 projection progress (2103.08624), 6 hover, 7 fly-thru-gate, "
                   "8 bootstrapped vision racing (2403.12203), 9 champion-level racing (Nature 2023)")
    p.add_argument("--track", type=str, default="circle", help="circle (the reference's main) or another Waypoints track function, e.g. reaching")
    p.add_argument("--model_path", type=str, default=None, help="SB3-format archive for --run_type cont / saved")
    p.add_argument("--max_seconds", type=float, default=None, help="wall-clock cap of run_full_training")
    p.add_argument("--minibatch", type=int, default=None, help="PPO minibatch size (default: rollout size / 32, at least 512)")
    p.add_argument("--n_epochs", type=int, default=10)
    p.add_argument("--tensorboard", type=str, default=None, help="directory for TensorBoard scalars (SB3 tag names)")
    p.add_argument("--rollout_steps", type=int, default=None, help="steps per env per PPO rollout (default: n_steps=4096 / scaled)")
    p.add_argument("--rollout_impl", type=str, default="torch", choices=["torch", "fused"],
                   help="rollout collection: torch (per-step host loop, torch.Generator noise) or fused (Philox noise keyed by the "
                        "global env id, collection replayed from a CUDA graph). PPO: dn_ppo_act, needs the fused PPO handle; SAC: "
                        "dn_sac_act, needs a compute-capability-10 device (the SAC gradient step stays on torch)")
    return p


def parse_args(argv=None):
    return build_parser().parse_args(argv)
