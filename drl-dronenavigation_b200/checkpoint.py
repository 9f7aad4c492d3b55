"""SB3-format checkpoint I/O for the PPO and SAC learners (SURVEY.md section 8 f.2).

The reference saves and reloads Stable-Baselines3 archives -- ``best_model.zip`` / ``success_model.zip`` written by
``EvalCallback`` / ``model.save`` (Sol/Model/PBDroneSimulator.py:719-746) and read back by ``PPO.load`` in
``test_saved`` (:438-572) and ``run_full(cont)`` (:132-134).  An SB3 archive is a zip with

    data                          JSON of the constructor arguments (spaces etc. as base64 cloudpickle)
    policy.pth                    torch state_dict of the ActorCriticPolicy
    policy.optimizer.pth          torch state_dict of its Adam optimiser
    pytorch_variables.pth         extra tensors (none for PPO)
    _stable_baselines3_version    text
    system_info.txt               text

This module reads ``policy.pth`` (and the optimiser, when present) of such an archive into the torch-native
``ActorCritic`` of ``ppo.py`` and writes archives with the same member names and the same ``policy.pth`` key names, so
policies move in both directions:  reference-trained ``*.zip`` -> GPU environment, and a policy trained here ->
``ActorCriticPolicy.load_state_dict(torch.load(zf.open("policy.pth")))`` in an SB3 installation.  The ``data`` member
written here is plain JSON of the hyper-parameters (no cloudpickled spaces: gymnasium is not installable in this
image), which ``PPO.load`` needs ``custom_objects`` for; the tensor members are exact.

Key map for ``net_arch=dict(pi=[512, 512, 256], vf=[512, 512, 256])``, ``share_features_extractor=False``
(PBDroneSimulator.py:251-258; SB3 MlpExtractor / ActorCriticPolicy naming):

    mlp_extractor.policy_net.{0,2,4}.{weight,bias}  <->  pi.{0,2,4}.{weight,bias}
    action_net.{weight,bias}                        <->  pi.6.{weight,bias}
    mlp_extractor.value_net.{0,2,4}.{weight,bias}   <->  vf.{0,2,4}.{weight,bias}
    value_net.{weight,bias}                         <->  vf.6.{weight,bias}
    log_std                                         <->  log_std

SAC (``SAC.load(self.continued_agent)`` / ``model.save``, PBDroneSimulator.py:355-362,741-746; hyper-parameters :290-331).  An SB3
SAC archive holds ``policy.pth`` (SACPolicy: actor, critic, critic_target), ``actor.optimizer.pth``, ``critic.optimizer.pth``,
``ent_coef_optimizer.pth`` and ``pytorch_variables.pth`` = ``{"log_ent_coef": tensor}``.  Key map for
``net_arch=dict(pi=[256, 256], qf=[256, 256, 128])``:

    actor.latent_pi.{0,2}.{weight,bias}             <->  actor.latent.{0,2}.{weight,bias}
    actor.mu / actor.log_std .{weight,bias}         <->  actor.mu / actor.log_std
    critic.qf{i}.{0,2,4,6}.{weight,bias}            <->  critic.qs.{i}.{0,2,4,6}.{weight,bias}
    critic_target.qf{i}.{0,2,4,6}.{weight,bias}     <->  critic_target.qs.{i}.{0,2,4,6}.{weight,bias}

The replay buffer the reference's ``SaveReplayBufferCallback`` writes (``Sol/Utilities/Callbacks.py:13-39``:
``model.save_replay_buffer(".../replay_buffer.pkl")``) is SB3's pickled ``ReplayBuffer`` object; without SB3 in this image the
file written here is a pickled dict with that object's attribute names (``observations``, ``next_observations``, ``actions``,
``rewards``, ``dones``, ``pos``, ``full``, ``buffer_size``, ``n_envs``) and the loader accepts either (see ``sac.ReplayBuffer``).
"""
from __future__ import annotations

import io
import json
import zipfile
from typing import Dict, Optional

import torch

SB3_VERSION_TAG = "2.3.2"        # written to _stable_baselines3_version (format unchanged since SB3 1.x)


def _key_map(n_hidden_pi: int, n_hidden_vf: int) -> Dict[str, str]:
    """ours -> SB3."""
    m = {"log_std": "log_std"}
    for ours, theirs, head, n in (("pi", "policy_net", "action_net", n_hidden_pi), ("vf", "value_net", "value_net", n_hidden_vf)):
        for layer in range(n):
            for leaf in ("weight", "bias"):
                m[f"{ours}.{2 * layer}.{leaf}"] = f"mlp_extractor.{theirs}.{2 * layer}.{leaf}"
        for leaf in ("weight", "bias"):
            m[f"{ours}.{2 * n}.{leaf}"] = f"{head}.{leaf}"
    return m


def _sb3_param_order(n_hidden_pi: int, n_hidden_vf: int):
    """SB3 names in the order of ``ActorCriticPolicy.parameters()`` -- the positional index of ``policy.optimizer.pth``:
    log_std, mlp_extractor.policy_net.*, mlp_extractor.value_net.*, action_net.*, value_net.* (checked against the archive SB3
    itself wrote, Sol/pyfly/ppo_quadx_waypoints.zip)."""
    names = ["log_std"]
    for net, n in (("policy_net", n_hidden_pi), ("value_net", n_hidden_vf)):
        for layer in range(n):
            names += [f"mlp_extractor.{net}.{2 * layer}.weight", f"mlp_extractor.{net}.{2 * layer}.bias"]
    return names + ["action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias"]


def policy_to_sb3_state_dict(policy) -> Dict[str, torch.Tensor]:
    sd = policy.state_dict()
    n_pi = sum(1 for k in sd if k.startswith("pi.") and k.endswith(".weight")) - 1
    n_vf = sum(1 for k in sd if k.startswith("vf.") and k.endswith(".weight")) - 1
    km = _key_map(n_pi, n_vf)
    return {km[k]: v.detach().cpu().clone() for k, v in sd.items()}


def sb3_state_dict_to_policy(policy, sb3_sd: Dict[str, torch.Tensor], strict: bool = True) -> None:
    sd = policy.state_dict()
    n_pi = sum(1 for k in sd if k.startswith("pi.") and k.endswith(".weight")) - 1
    n_vf = sum(1 for k in sd if k.startswith("vf.") and k.endswith(".weight")) - 1
    km = _key_map(n_pi, n_vf)
    new = {}
    for ours, theirs in km.items():
        if theirs not in sb3_sd:
            if strict:
                raise KeyError(f"{theirs} missing from the SB3 policy state_dict (has: {sorted(sb3_sd)[:6]} ...)")
            continue
        t = sb3_sd[theirs]
        if tuple(t.shape) != tuple(sd[ours].shape):
            raise ValueError(f"{theirs}: shape {tuple(t.shape)} does not match this policy's {tuple(sd[ours].shape)} "
                             "(net_arch differs from PBDroneSimulator.py:251-258?)")
        new[ours] = t.to(sd[ours].device, sd[ours].dtype)
    extra = [k for k in sb3_sd if k not in km.values() and not k.startswith(("features_extractor", "pi_features_extractor",
                                                                              "vf_features_extractor"))]
    if strict and extra:
        raise KeyError(f"unexpected keys in the SB3 policy state_dict: {extra[:6]}")
    policy.load_state_dict(new, strict=strict)


def _save_tensor_member(zf: zipfile.ZipFile, name: str, obj) -> None:
    buf = io.BytesIO()
    torch.save(obj, buf)
    zf.writestr(name, buf.getvalue())


def save_sb3_zip(path: str, learner, extra: Optional[dict] = None) -> str:
    """Writes an SB3-layout archive of a ``PPOLearner`` (policy + Adam state + hyper-parameters); a ``SACLearner`` goes to
    :func:`save_sb3_sac_zip`."""
    if hasattr(learner, "actor") and hasattr(learner, "critic_target"):
        return save_sb3_sac_zip(path, learner, extra)
    cfg = learner.cfg
    sd = policy_to_sb3_state_dict(learner.policy)
    km = _key_map(len(cfg.pi_arch), len(cfg.vf_arch))
    # SB3's optimiser state_dict indexes parameters by position in ITS policy.parameters() (log_std first, then the two
    # extractor nets, then the heads): re-index ours (pi.*, vf.*, log_std) into that order so that SB3's
    # optimizer.load_state_dict attaches every Adam moment to the parameter it belongs to; the names are recorded as well
    opt_sd = learner.opt.state_dict()
    ours_names = [km[n] for n, _ in learner.policy.named_parameters()]
    sb3_order = _sb3_param_order(len(cfg.pi_arch), len(cfg.vf_arch))
    pos_ours = {nm: i for i, nm in enumerate(ours_names)}
    groups = [dict(g) for g in opt_sd["param_groups"]]
    for g in groups:
        g["params"] = list(range(len(sb3_order)))
    opt_state = {"state": {j: {k: (v.detach().cpu().clone() if torch.is_tensor(v) else v) for k, v in opt_sd["state"][pos_ours[nm]].items()}
                           for j, nm in enumerate(sb3_order) if pos_ours[nm] in opt_sd["state"]},
                 "param_groups": groups,
                 "param_names": sb3_order}
    data = {"policy_class": "stable_baselines3.common.policies.ActorCriticPolicy", "algo": "PPO",
            "n_steps": cfg.n_steps, "batch_size": cfg.batch_size, "n_epochs": cfg.n_epochs, "gamma": cfg.gamma,
            "gae_lambda": cfg.gae_lambda, "ent_coef": cfg.ent_coef, "vf_coef": cfg.vf_coef, "clip_range": cfg.clip_range,
            "clip_range_vf": cfg.clip_range_vf, "normalize_advantage": cfg.normalize_advantage,
            "max_grad_norm": cfg.max_grad_norm, "target_kl": cfg.target_kl, "learning_rate": cfg.learning_rate,
            "policy_kwargs": {"activation_fn": "torch.nn.Tanh", "net_arch": {"pi": list(cfg.pi_arch), "vf": list(cfg.vf_arch)},
                              "share_features_extractor": False, "log_std_init": cfg.log_std_init},
            "observation_space": {"type": "Box", "shape": [learner.policy.pi[0].in_features], "dtype": "float32"},
            "action_space": {"type": "Box", "low": -1.0, "high": 1.0, "shape": [learner.policy.log_std.numel()], "dtype": "float32"},
            "n_updates": learner.n_updates, "seed": cfg.seed, "written_by": "drl_dronenavigation_b200"}
    if extra:
        data.update(extra)
    if not path.endswith(".zip"):
        path += ".zip"
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as zf:
        zf.writestr("data", json.dumps(data, indent=2))
        _save_tensor_member(zf, "policy.pth", sd)
        _save_tensor_member(zf, "policy.optimizer.pth", opt_state)
        _save_tensor_member(zf, "pytorch_variables.pth", None)
        zf.writestr("_stable_baselines3_version", SB3_VERSION_TAG)
        zf.writestr("system_info.txt", f"torch {torch.__version__}\n")
    return path


def load_sb3_zip(path: str, learner, load_optimizer: bool = False, strict: bool = True) -> dict:
    """Loads ``policy.pth`` of an SB3 archive (the reference's ``best_model.zip``) into ``learner.policy``.
    Returns the parsed ``data`` member (or {} when it is not plain JSON-decodable).  A ``SACLearner`` goes to :func:`load_sb3_sac_zip`."""
    if hasattr(learner, "actor") and hasattr(learner, "critic_target"):
        return load_sb3_sac_zip(path, learner, load_optimizer=load_optimizer, strict=strict)
    with zipfile.ZipFile(path) as zf:
        names = set(zf.namelist())
        if "policy.pth" not in names:
            raise KeyError(f"{path}: no policy.pth member (members: {sorted(names)})")
        sb3_sd = torch.load(io.BytesIO(zf.read("policy.pth")), map_location="cpu", weights_only=True)
        sb3_state_dict_to_policy(learner.policy, sb3_sd, strict=strict)
        if load_optimizer and "policy.optimizer.pth" in names:
            opt = torch.load(io.BytesIO(zf.read("policy.optimizer.pth")), map_location="cpu", weights_only=False)
            # SB3 orders parameters as ITS policy.parameters() does (log_std, policy_net, value_net, action_net, value_net head);
            # ours: pi..., vf..., log_std.  Re-index by name: the recorded names when this repo wrote the archive, SB3's known
            # order otherwise (every genuine SB3 archive); a state that does not fit is dropped LOUDLY, never silently
            import warnings
            params = list(learner.policy.named_parameters())
            names_theirs = opt.get("param_names") or _sb3_param_order(len(learner.cfg.pi_arch), len(learner.cfg.vf_arch))
            km = _key_map(len(learner.cfg.pi_arch), len(learner.cfg.vf_arch))
            order = {km[n]: i for i, (n, _) in enumerate(params)}
            state, ok = {}, len(names_theirs) == len(params) and set(names_theirs) == set(order)
            if ok:
                for j, nm in enumerate(names_theirs):
                    if j in opt.get("state", {}):
                        st = opt["state"][j]
                        if tuple(st["exp_avg"].shape) != tuple(params[order[nm]][1].shape):
                            ok = False
                            break
                        state[order[nm]] = st
            if ok and state:
                learner.load_optimizer_state(state)
            else:
                warnings.warn(f"{path}: the optimiser state does not match this policy's parameters and was NOT loaded "
                              "(Adam restarts from zero moments)", RuntimeWarning)
        data = {}
        if "data" in names:
            try:
                data = json.loads(zf.read("data").decode())
            except Exception:  # noqa: BLE001
                data = {}
    return data


# ---------------------------------------------------------------------------------------------------------------------
# SAC
# ---------------------------------------------------------------------------------------------------------------------
def _sac_key(ours: str) -> str:
    """name in SACLearner's modules ("actor.latent.0.weight", "critic.qs.1.4.bias") -> SB3 SACPolicy key."""
    parts = ours.split(".")
    if parts[0] == "actor" and parts[1] == "latent":
        parts[1] = "latent_pi"
    elif parts[0] in ("critic", "critic_target") and parts[1] == "qs":
        parts[1:3] = [f"qf{parts[2]}"]
    return ".".join(parts)


def _sac_modules(learner):
    return (("actor", learner.actor), ("critic", learner.critic), ("critic_target", learner.critic_target))


def sac_to_sb3_state_dict(learner) -> Dict[str, torch.Tensor]:
    return {_sac_key(f"{pre}.{k}"): v.detach().cpu().clone() for pre, mod in _sac_modules(learner) for k, v in mod.state_dict().items()}


def sb3_state_dict_to_sac(learner, sb3_sd: Dict[str, torch.Tensor], strict: bool = True) -> None:
    used = set()
    for pre, mod in _sac_modules(learner):
        own = mod.state_dict()
        new = {}
        for k, v in own.items():
            theirs = _sac_key(f"{pre}.{k}")
            if theirs not in sb3_sd:
                if strict:
                    raise KeyError(f"{theirs} missing from the SB3 SAC policy state_dict (has: {sorted(sb3_sd)[:6]} ...)")
                continue
            t = sb3_sd[theirs]
            if tuple(t.shape) != tuple(v.shape):
                raise ValueError(f"{theirs}: shape {tuple(t.shape)} does not match this learner's {tuple(v.shape)} "
                                 "(net_arch differs from PBDroneSimulator.py:296-300?)")
            new[k] = t.to(v.device, v.dtype)
            used.add(theirs)
        mod.load_state_dict(new, strict=strict)
    extra = [k for k in sb3_sd if k not in used and "features_extractor" not in k]
    if strict and extra:
        raise KeyError(f"unexpected keys in the SB3 SAC policy state_dict: {extra[:6]}")


def _opt_cpu(opt) -> dict:
    sd = opt.state_dict()
    return {"state": {i: {k: (v.detach().cpu() if torch.is_tensor(v) else v) for k, v in st.items()} for i, st in sd["state"].items()},
            "param_groups": sd["param_groups"]}


def save_sb3_sac_zip(path: str, learner, extra: Optional[dict] = None) -> str:
    """Writes an SB3-layout archive of a ``SACLearner``: SB3's member names, SACPolicy's key names, parameter order of the
    optimisers = ``actor.parameters()`` / ``critic.parameters()`` as in SB3 (latent layers, then mu, then log_std; qf0, then qf1)."""
    cfg = learner.cfg
    data = {"policy_class": "stable_baselines3.sac.policies.SACPolicy", "algo": "SAC", "batch_size": cfg.batch_size,
            "buffer_size": cfg.buffer_size, "learning_starts": cfg.learning_starts, "train_freq": cfg.train_freq,
            "gradient_steps": cfg.gradient_steps, "tau": cfg.tau, "gamma": cfg.gamma, "learning_rate": cfg.learning_rate,
            "target_update_interval": cfg.target_update_interval, "ent_coef": "auto", "target_entropy": learner.target_entropy,
            "policy_kwargs": {"activation_fn": "torch.nn.ReLU", "net_arch": {"pi": list(cfg.pi_arch), "qf": list(cfg.qf_arch)},
                              "n_critics": cfg.n_critics, "share_features_extractor": False},
            "observation_space": {"type": "Box", "shape": [learner.actor.latent[0].in_features], "dtype": "float32"},
            "action_space": {"type": "Box", "low": -1.0, "high": 1.0, "shape": [learner.actor.mu.out_features], "dtype": "float32"},
            "n_updates": learner.n_updates, "seed": cfg.seed, "written_by": "drl_dronenavigation_b200"}
    if extra:
        data.update(extra)
    if not path.endswith(".zip"):
        path += ".zip"
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as zf:
        zf.writestr("data", json.dumps(data, indent=2))
        _save_tensor_member(zf, "policy.pth", sac_to_sb3_state_dict(learner))
        _save_tensor_member(zf, "actor.optimizer.pth", _opt_cpu(learner.actor_opt))
        _save_tensor_member(zf, "critic.optimizer.pth", _opt_cpu(learner.critic_opt))
        _save_tensor_member(zf, "ent_coef_optimizer.pth", _opt_cpu(learner.ent_opt))
        _save_tensor_member(zf, "pytorch_variables.pth", {"log_ent_coef": learner.log_ent_coef.detach().cpu().clone()})
        zf.writestr("_stable_baselines3_version", SB3_VERSION_TAG)
        zf.writestr("system_info.txt", f"torch {torch.__version__}\n")
    return path


def load_sb3_sac_zip(path: str, learner, load_optimizer: bool = False, strict: bool = True) -> dict:
    """Loads an SB3 SAC archive (``SAC.load`` of the reference's ``--run_type cont``, PBDroneSimulator.py:355-357) into a ``SACLearner``."""
    with zipfile.ZipFile(path) as zf:
        names = set(zf.namelist())
        if "policy.pth" not in names:
            raise KeyError(f"{path}: no policy.pth member (members: {sorted(names)})")
        sb3_state_dict_to_sac(learner, torch.load(io.BytesIO(zf.read("policy.pth")), map_location="cpu", weights_only=True), strict=strict)
        if "pytorch_variables.pth" in names:
            pv = torch.load(io.BytesIO(zf.read("pytorch_variables.pth")), map_location="cpu", weights_only=False)
            if isinstance(pv, dict) and pv.get("log_ent_coef") is not None:
                with torch.no_grad():
                    learner.log_ent_coef.copy_(pv["log_ent_coef"].reshape(learner.log_ent_coef.shape).to(learner.log_ent_coef.device))
        if load_optimizer:
            members = {"actor": "actor.optimizer.pth", "critic": "critic.optimizer.pth", "ent_coef": "ent_coef_optimizer.pth"}
            learner.load_optimizer_state({name: torch.load(io.BytesIO(zf.read(m)), map_location="cpu", weights_only=False)
                                          for name, m in members.items() if m in names})
        data = {}
        if "data" in names:
            try:
                data = json.loads(zf.read("data").decode())
            except Exception:  # noqa: BLE001
                data = {}
    return data
