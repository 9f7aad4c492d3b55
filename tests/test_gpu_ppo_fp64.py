"""The fused PPO update (include/dnppo.h) stage by stage against the FP64 reference (tests/ppo_fp64_reference.py), at every
shape the trainer and the ABI reach.

Per configuration, one minibatch at a time through the C ABI (begin_update / minibatch_grad / minibatch_apply), three
minibatches in a row (Adam's bias corrections at t = 1, 2, 3), each from the handle's current parameters and on fresh rows:
  1. the gathered observation planes (hi + lo = the rows to BF16-pair precision, padding columns exactly 0);
  2. every hidden activation h_l of both nets;
  3. every pre-activation gradient dz_l (layer L isolates the head kernel, l < L each dgrad);
  4. the flat gradient bucket, tensor by tensor;
  5. the loss statistics and the KL early-stop vote;
then, from the kernel's OWN bucket, clip_grad_norm_ + Adam in FP64 against minibatch_apply: parameters, moments, the
gradient norm and the refreshed BF16 weight planes.

Rollouts carry branch margins (every ratio > delta relative from 1 +- clip_range, every value change > delta from
+- clip_range_vf): the kernels take every clipping branch the reference takes, the clip fraction must match exactly, and no
bound absorbs flipped samples.  Bounds, bf16x3 (BF16 hi + lo planes, three products; the dropped lo x lo term and the rounding
of lo are ~2^-17 of |a||b| per product, DESIGN.md section 4b):
  * activations 5e-5 absolute (|h| <= 1; each layer adds a few 2^-18 roundings of its operands and output and carries the
    input error through a weight row of norm sqrt(2); measured maxima over 10^6..10^7 entries: 2e-5 at depth 3 and 4);
  * dz_l 5e-5 max-norm relative (per-sample quantities);
  * every gradient tensor 5e-5 of the largest SUM OF MAGNITUDES of its per-sample contributions (|dZ|^T |H|, sum |dZ|): a
    gradient is a sum over the rows whose terms cancel (value errors v - ret of both signs), while the per-sample errors
    share a component (the rounding of the weights is the same for every row) that adds up coherently -- measured against
    max |gradient| instead, the value net's biases at 2048 rows reach 2e-4 while their per-sample inputs dz are good to 1e-5.
    The denominator is floored at 1e-3 of the largest gradient entry of the network (log_std: data term - ent_coef);
  * loss statistics 1e-5 relative to the mean magnitude of their per-sample terms;
  * Adam: |dparam| <= 1e-5 lr + half an ulp (the kernel's FP32 step is a few roundings of a quantity <= lr, rsqrtf and
    powf add a few ulp), moments 1e-5 relative, the gradient norm 1e-6 relative (summed in FP64 on the device).  The
    reference takes the hyper-parameters as dn_ppo_config carries them, in FP32: 0.999f = 0.999 + 1.3e-8, so 1 - beta2 is
    1.3e-5 (relative) below 0.001 and exp_avg_sq is as much below torch.optim.Adam's (which weights g^2 by 1 - 0.999 in
    double); the bias correction 1 - beta2^t shares the factor, so the parameters agree to ~1e-7 lr either way.
bf16 (hi planes only): 3e-2 max-norm relative for every stage, the per-contraction bound of tests/test_gpu_mlp.py compounded
over the depth; its margins are 3e-2 since its logits move by more than 1e-3.
"""
import pytest
import torch

from tests import ppo_fp64_reference as R

pytestmark = pytest.mark.gpu


def _cc10():
    return torch.cuda.is_available() and torch.cuda.get_device_capability()[0] == 10


A3 = (512, 512, 256)
# id: (obs_dim, act_dim, pi_arch, vf_arch, minibatch B, handle rows max_rows, PPOConfig overrides, test options)
CONFIGS = {
    "bench": (13, 4, A3, A3, 32768, 65536, dict(target_kl=0.05), {}),
    "obs12": (12, 4, A3, A3, 4096, 4096, {}, {}),
    "mb128": (13, 4, A3 + (128,), A3 + (128,), 128, 4096, {}, {}),
    "mb1280": (13, 4, A3, A3, 1280, 2560, {}, {}),
    "mb1152": (13, 4, A3, A3, 1152, 2304, {}, {}),        # a multiple of 128 but not of 256: single-CTA tiles (M = 128)
    "act1": (13, 1, (256, 128), (256, 128), 1024, 1024, {}, {}),
    "act3": (13, 3, (256, 128), (256, 128), 1024, 1024, dict(target_kl=0.01), {}),
    "unequal-depth": (13, 4, (256, 128), A3, 2048, 2048, {}, {}),
    "unequal-width": (13, 4, (512, 256), (256, 512), 2048, 2048, {}, {}),
    "head512": (13, 4, (512, 512), (512, 512), 2048, 2048, {}, {}),
    "head384": (13, 4, (256, 384), (128,), 1024, 1024, {}, {}),
    "options": (13, 4, (256, 128), (256, 128), 1024, 1024,
                dict(clip_range_vf=None, normalize_advantage=False, ent_coef=0.0, max_grad_norm=1e9), {}),
    "world2": (13, 4, (256, 128), (256, 128), 1024, 1024, {}, dict(world=2)),
    "bf16": (13, 4, A3, A3, 4096, 4096, dict(mlp_precision="bf16"), {}),
}


def _build(cid, monkeypatch):
    """A fused learner with non-zero biases and log_std, its handle sized by a forward of max_rows rows (as the trainer's
    rollout forward sizes it), and a rollout of max(max_rows, 2 B) rows."""
    from drl_dronenavigation_b200 import ppo
    obs_dim, act_dim, pi, vf, B, max_rows, over, opt = CONFIGS[cid]
    kw = dict(pi_arch=pi, vf_arch=vf, batch_size=B, cuda_graph=False, update_impl="fused", target_kl=None, matmul_precision="fp32")
    kw.update(over)
    L = ppo.PPOLearner(obs_dim, act_dim, ppo.PPOConfig(**kw), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(5)
    with torch.no_grad():
        for p in L.params:
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, device="cuda", generator=g))
    spec = R.Spec(obs_dim, act_dim, pi, vf)
    ro = R.make_rollout(L.flat_parameters(), spec, max(max_rows, 2 * B), seed=B + act_dim, device="cuda")
    with monkeypatch.context() as m:
        if opt.get("world"):
            m.setattr(ppo, "_world", lambda: opt["world"])     # the handle is configured for world_size ranks
        L.forward(ro[0][:max_rows])
    assert L.fused is not None and L.fused.max_rows == max_rows and L.fused.cfg_c.world_size == opt.get("world", 1)
    return L, spec, ro


def _c_rollout(L, ro):
    r = L.fused.L.dn_ppo_rollout()
    r.obs, r.actions, r.old_log_prob, r.old_values, r.advantages, r.returns = [t.data_ptr() for t in ro]
    return r


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
@pytest.mark.parametrize("cid", list(CONFIGS))
def test_minibatch_stages_match_fp64(cid, monkeypatch):
    obs_dim, act_dim, pi, vf, B, max_rows, over, opt = CONFIGS[cid]
    L, spec, ro = _build(cid, monkeypatch)
    cfg, fu = L.cfg, L.fused
    world = opt.get("world", 1)
    bf16 = cfg.mlp_precision == "bf16"
    tol_h, tol_g, tol_s = (3e-2, 3e-2, 3e-2) if bf16 else (5e-5, 5e-5, 1e-5)
    delta = 3e-2 if bf16 else 1e-3
    plane_rel = 2.0 ** -8 if bf16 else 2.0 ** -16          # BF16 (RN) / BF16 pair representation of an FP32 value
    lr = cfg.learning_rate
    r = _c_rollout(L, ro)
    gen = torch.Generator(device="cuda").manual_seed(17)
    report = {}
    try:
        for k in range(3):
            flat = L.flat_parameters()
            idx = torch.randperm(ro[0].shape[0], device="cuda", generator=gen)[:B]
            info = R.enforce_margins(flat, spec, ro, idx, cfg.clip_range, cfg.clip_range_vf, delta)
            ref = R.minibatch(flat, spec, [t[idx] for t in ro], cfg.clip_range, cfg.clip_range_vf, cfg.normalize_advantage,
                              cfg.ent_coef, cfg.vf_coef)
            fu.begin_update()                    # statistics of this minibatch alone
            fu.minibatch_grad(r, idx)
            torch.cuda.synchronize()
            err = {}
            # 1. gathered observations
            x = fu.buffer("x", B, 64)
            rows = ro[0][idx].double()
            assert torch.all(x[:, obs_dim:] == 0), cid
            err["x"] = float(((x[:, :obs_dim].double() - rows).abs() / rows.abs().clamp_min(1e-30)).max())
            assert err["x"] <= plane_rel, err
            # 2. activations, 3. pre-activation gradients
            for net, arch in (("pi", pi), ("vf", vf)):
                for l, w in enumerate(arch, start=1):
                    err[f"{net}.h{l}"] = (R.max_rel(fu.buffer(f"{net}.h{l}", B, w), ref[f"h_{net}"][l - 1]) if bf16 else
                                          float((fu.buffer(f"{net}.h{l}", B, w).double() - ref[f"h_{net}"][l - 1]).abs().max()))
                    err[f"{net}.dz{l}"] = R.max_rel(fu.buffer(f"{net}.dz{l}", B, w), ref[f"dz_{net}"][l - 1])
            # 4. the bucket, tensor by tensor
            gerr, floored = R.per_tensor_errors(L._flat, ref["grad"], spec, scale=ref["grad_magnitude"])
            plain = max(R.per_tensor_errors(L._flat, ref["grad"], spec)[0].values())      # for the log: vs max |gradient|
            # 5. statistics and the vote
            st = fu.stats()
            got = {"policy_gradient_loss": st.policy_gradient_loss, "value_loss": st.value_loss, "approx_kl": st.approx_kl}
            serr = {s: abs(got[s] - ref["stats"][s]) / max(abs(ref["stats"][s]), ref["stat_scale"][s]) for s in got}
            print(f"\n{cid} minibatch {k + 1}: margins {info}")
            print("  stages", {s: f"{e:.1e}" for s, e in err.items()})
            print("  grad", {s: f"{e:.1e}" for s, e in gerr.items()}, "floored:", floored)
            print("  stats", {s: f"{e:.1e}" for s, e in serr.items()}, "clipped", ref["n_clipped"], "of", B,
                  f"(gradient vs max |gradient|: {plain:.1e})")
            for s, e in err.items():
                assert e <= (tol_h if ".h" in s else tol_g), (cid, k, s, e)
            assert max(gerr.values()) <= tol_g, (cid, k, gerr)
            assert max(serr.values()) <= tol_s, (cid, k, serr)
            assert round(st.clip_fraction * B) == ref["n_clipped"] and abs(st.clip_fraction * B - ref["n_clipped"]) < 1e-9
            assert st.minibatches == 1
            vote = float(L._bucket[-1])
            if cfg.target_kl is None:
                assert vote == 0.0
            else:
                limit = 1.5 * cfg.target_kl
                assert abs(ref["stats"]["approx_kl"] - limit) > 1e-3 * limit     # decided far beyond the kernel's error
                assert vote == float(ref["stats"]["approx_kl"] > limit), (vote, ref["stats"]["approx_kl"], limit)
            # ---- clip + Adam from the kernel's own bucket ----
            if world > 1:
                L._bucket.mul_(world)            # the all-reduce of `world` identical ranks: a sum, vote included
                assert float(L._bucket[-1]) == world * vote
            L._bucket[-1] = 0.0                  # this comparison is of a step that is taken
            grad = L._flat.clone()
            p0, m0, v0, step = fu.params.clone(), fu.exp_avg.clone(), fu.exp_avg_sq.clone(), float(fu.step)
            assert step == k
            c = fu.cfg_c                         # FP32 hyper-parameters, as the handle holds them
            p_ref, m_ref, v_ref, norm = R.clip_adam(grad, p0, m0, v0, step, lr=c.learning_rate, max_grad_norm=c.max_grad_norm,
                                                    world_size=world, beta1=c.beta1, beta2=c.beta2, eps=c.adam_eps)
            fu.minibatch_apply()
            st = fu.stats()
            assert st.optimizer_steps == 1 and float(fu.step) == k + 1
            excess = float(((fu.params.double() - p_ref).abs() - R.half_ulp(fu.params)).max())
            aerr = {"param (lr)": excess / lr, "exp_avg": R.max_rel(fu.exp_avg, m_ref), "exp_avg_sq": R.max_rel(fu.exp_avg_sq, v_ref),
                    "norm": abs(st.last_grad_norm - norm) / norm}
            print("  adam", {s: f"{e:.1e}" for s, e in aerr.items()}, f"norm {norm:.3f} (clip at {cfg.max_grad_norm})")
            assert aerr["param (lr)"] <= 1e-5 and aerr["exp_avg"] <= 1e-5 and aerr["exp_avg_sq"] <= 1e-5, (cid, k, aerr)
            assert aerr["norm"] <= 1e-6, (cid, k, aerr)
            # the BF16 weight planes follow the new parameters (layer 1: zero padding columns obs_dim..63)
            P = R.split(fu.params, spec)
            for net, arch in (("pi", pi), ("vf", vf)):
                for l, w in enumerate(arch, start=1):
                    cols = obs_dim if l == 1 else arch[l - 2]
                    ld = 64 if l == 1 else cols
                    planes = fu.buffer(f"{net}.w{l}", w, ld)
                    wt = P[f"{net}.{2 * (l - 1)}.weight"].double()
                    assert torch.all(planes[:, cols:] == 0)
                    assert float(((planes[:, :cols].double() - wt).abs() - plane_rel * wt.abs()).max()) <= 0, (net, l)
            for s, e in {**err, **gerr, **serr, **aerr}.items():
                report[s] = max(report.get(s, 0.0), e)
            report["grad vs max|grad|"] = max(report.get("grad vs max|grad|", 0.0), plain)
        print(f"{cid} maxima over 3 minibatches:", {s: f"{e:.1e}" for s, e in report.items()})
    finally:
        fu.close()


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
@pytest.mark.parametrize("cid", list(CONFIGS))
def test_forward_matches_fp64_and_replanning_is_invisible(cid, monkeypatch):
    """dn_ppo_forward at 1, 127, 129 and max_rows rows against FP64 (mean and value within 2e-5 of max(1, max |ref|); bf16:
    3e-2), between two gradients of the same minibatch: every row count re-plans the contractions (tile shapes, wgrad slices,
    grid sizes) and the second gradient re-builds the reduction table, yet the two buckets are BIT-identical, because every
    plan and table is a function of the row count alone."""
    obs_dim, act_dim, pi, vf, B, max_rows, over, opt = CONFIGS[cid]
    L, spec, ro = _build(cid, monkeypatch)
    fu = L.fused
    tol = 3e-2 if L.cfg.mlp_precision == "bf16" else 2e-5
    r = _c_rollout(L, ro)
    idx = torch.randperm(ro[0].shape[0], device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))[:B]
    try:
        fu.begin_update()
        fu.minibatch_grad(r, idx)
        first = L._bucket.clone()
        flat = L.flat_parameters()
        errs = {}
        for rows in (max_rows, 1, 127, 129):
            mean, value = fu.forward(ro[0][:rows])
            m_ref, v_ref = R.policy(flat, spec, ro[0][:rows])
            errs[rows] = (float((mean.double() - m_ref).abs().max()) / max(1.0, float(m_ref.abs().max())),
                          float((value.double() - v_ref).abs().max()) / max(1.0, float(v_ref.abs().max())))
        print(f"\n{cid} forward (mean, value) errors by rows:", {k: f"{a:.1e} {b:.1e}" for k, (a, b) in errs.items()})
        assert max(max(e) for e in errs.values()) <= tol, errs
        fu.minibatch_grad(r, idx)
        assert torch.equal(first, L._bucket), float((first - L._bucket).abs().max())
    finally:
        fu.close()


@pytest.mark.skipif(not _cc10(), reason="needs an sm_100 device")
def test_hidden_width_above_512_trains_on_the_torch_path():
    """A 1024-wide hidden layer is beyond what dn_ppo_create accepts: update_impl="auto" keeps the torch path from the start."""
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOLearner
    arch = (1024, 512, 256)
    L = PPOLearner(13, 4, PPOConfig(pi_arch=arch, vf_arch=arch, batch_size=256, n_epochs=1, target_kl=None), device="cuda")
    assert not L.want_fused
    obs = torch.randn(512, 13, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    act, logp, v = L.act(obs)
    p0 = L.flat_parameters().clone()
    out = L.update(obs, act, logp, v, torch.randn_like(v), v + 1.0)
    assert L.fused is None and out["minibatches"] == 2 and "impl" not in out
    assert not torch.equal(p0, L.flat_parameters())
    with pytest.raises(RuntimeError, match="between 128 and 512"):
        PPOLearner(13, 4, PPOConfig(pi_arch=arch, vf_arch=arch, update_impl="fused"), device="cuda")
