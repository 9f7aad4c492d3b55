"""The gradient all-reduce over peer memory (include/dnppo.h: dn_ppo_comm_create / _connect / dn_ppo_allreduce;
csrc/ppo_comm.cuh) and the data-parallel fused PPO update around it, with real ranks.

Every case runs W rank processes (torch.multiprocessing.spawn, gloo for the host side; comm_setup gathers the IPC handles on CPU
tensors when the backend is not NCCL).  Placement "shared" puts every rank on device 0: CUDA IPC works between processes on one
device and, without MPS, the contexts are time-sliced, so a rank's wait completes once its peers get their slices (this does
not exercise NVLink).  Placement "distinct" puts rank r on device r and skips when fewer than W devices are visible.

Every wait of the exchange kernel traps after about a minute of polling, so no rank may be left waiting for a peer that will
not come:
  * each rank initialises CUDA and builds its learners, then all ranks agree through an all_reduce(MIN) of an "ok" flag, and
    exchanges start only if every rank is ready (otherwise every rank returns, and the parent skips -- a device in
    exclusive-process compute mode refuses the second context -- or fails with the reported reasons);
  * every block of exchanges starts with dist.barrier(), as PPOLearner._update_fused does;
  * nothing between the first and the last exchange of a block asserts: results are recorded, and checked after the block or
    in the parent, which reads each rank's result dict from tmp_path.
The parent requests `built_lib`, so the children only load the library.

What is asserted (DESIGN.md section 6 and the dn_ppo_allreduce comment in include/dnppo.h):
  * the exchange leaves on every rank the rank-order FP32 sum ((g0 + g1) + g2) + ..., bit for bit (NaN payloads aside), for
    buckets of 4234, 73 610 and 803 594 floats (n mod 4W != 0: the tail of publish and collect), wide-range values, lanes where
    another summation order gives another result (tests/peer_allreduce_inputs.py), signed zeros, subnormals, +-inf and NaN;
    nothing outside the bucket is written;
  * the vote element holds the exact count of voting ranks;
  * it is capturable in a CUDA graph: replays continue the epoch, and a rank that replays a graph while its peers launch
    directly takes part in the same exchange; two handles per process interleave their exchanges (flags and epochs are per
    handle);
  * every rank calls it the same number of times (allreduce_calls, launched minibatches, early stop);
  * one data-parallel minibatch through the C ABI: gradient sum within the FP64 bound of the single-rank stage test, the apply
    divides by world_size (Adam in FP64 on the exchanged bucket), a vote of one rank freezes every rank;
  * a rank that cannot use the exchange (DN_PPO_ALLREDUCE=nccl on that rank alone) sends every rank to the fallback, and the
    fallback path (two graphs around a host all_reduce) agrees with the rank-order sum.
Not tested: a missing peer (the trap) and the epoch wrap at 2^32 calls.
"""
import hashlib
import os
import socket
import time
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import peer_allreduce_inputs as I
from tests import ppo_fp64_reference as R

pytestmark = pytest.mark.gpu

WORLDS = (2, 3, 4)
PLACEMENTS = ("shared", "distinct")
# exchanged policies: (pi_arch, vf_arch), n = n_params + 1 and the grid of dn_ppo_allreduce on a 148-SM B200
ARCHS = {
    "128": (((128,), (128,)), 4234, 3),                                  # chunks shorter than the grid stride
    "256-128": (((256, 128), (256, 128)), 73610, 36),
    "bench": (((512, 512, 256), (512, 512, 256)), 803594, 148),          # grid-stride loops, the real 3.2 MB bucket
}
PAD = 256                          # sentinel floats on each side of the bucket (a multiple of 4: the kernel reads float4)
MODES = ("direct", "graph", "mixed")
CALLS_PER_BLOCK = 8                # per handle; 24 per handle over the three modes
SPEC = R.Spec(13, 4, (256, 128), (256, 128))


def _cc10():
    return torch.cuda.is_available() and torch.cuda.get_device_capability()[0] == 10


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _agree(ok: bool) -> bool:
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


def _blocks(n, world, sms):
    """The grid dn_ppo_allreduce launches (ppo_update.cu): one 512-thread CTA per 2048 padded floats, at most one per SM."""
    q = 4 * world
    n_pad = -(-n // q) * q
    return max(1, min(-(-(n_pad // 4) // 512), sms))


# ---- the rank processes ------------------------------------------------------------------------------------------------------
def _child(rank, world, port, tmp, placement, case):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), LOCAL_WORLD_SIZE=str(world))
    os.environ.pop("DN_PPO_ALLREDUCE", None)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(minutes=10))
    out = {"ready": False}
    try:
        why, state = "", None
        try:
            dev = torch.device("cuda", rank if placement == "distinct" else 0)
            torch.cuda.set_device(dev)
            torch.zeros(1, device=dev)
            torch.cuda.synchronize(dev)
            state = _SETUP[case](rank, world, dev)
        except Exception as e:  # noqa: BLE001 -- reported to the parent, after every rank has been told
            why = f"rank {rank}: {type(e).__name__}: {e}"
        if _agree(not why):
            out = _RUN[case](state, rank, world, dev)
            out["ready"] = True
            torch.cuda.synchronize(dev)
            dist.barrier()                     # no rank frees an exchange region before every rank's last exchange is done
        else:
            out["why"] = why
    finally:
        torch.save(out, os.path.join(tmp, f"rank{rank}.pt"))
        dist.destroy_process_group()


def _spawn(case, world, placement, tmp_path):
    if not _cc10():
        pytest.skip("needs an sm_100 device")
    if placement == "distinct" and torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs ({torch.cuda.device_count()} visible)")
    t0 = time.perf_counter()
    mp.spawn(_child, args=(world, _free_port(), str(tmp_path), placement, case), nprocs=world, join=True)
    res = [torch.load(os.path.join(tmp_path, f"rank{r}.pt"), weights_only=False) for r in range(world)]
    why = [r["why"] for r in res if r.get("why")]
    if not all(r["ready"] for r in res):
        if any("busy or unavailable" in w for w in why):
            pytest.skip(f"device refuses a second process (exclusive-process compute mode?): {why}")
        pytest.fail(f"ranks not ready: {why}")
    print(f"\n{case} W={world} {placement}: {time.perf_counter() - t0:.1f} s for {world} rank processes")
    return res


# ---- 2. the exchange kernel against the exact rank-order FP32 sum --------------------------------------------------------------
def _exchange_learner(arch, dev):
    """A fused learner whose bucket sits inside a larger sentinel-filled tensor (re-seated before the handle exists: the handle
    keeps the bucket's pointer)."""
    from drl_dronenavigation_b200 import ppo
    (pi, vf), n, _ = ARCHS[arch]
    L = ppo.PPOLearner(13, 4, ppo.PPOConfig(pi_arch=pi, vf_arch=vf, update_impl="fused", cuda_graph=False, target_kl=None),
                       device=dev)
    assert L.n_params + 1 == n, (arch, L.n_params)
    big = torch.from_numpy(np.full(n + 2 * PAD, I.SENTINEL_BITS, np.uint32).view(np.float32)).to(dev)
    L._bucket = big[PAD:PAD + n]
    L._flat = L._bucket[:L.n_params]
    off = 0
    for p in L.params:
        p.grad = L._flat[off:off + p.numel()].view_as(p)
        off += p.numel()
    fu = L.ensure_fused(128)
    assert fu.cfg_c.world_size == dist.get_world_size()
    return {"L": L, "fu": fu, "big": big, "n": n}


def _setup_exchange(rank, world, dev):
    return {arch: [_exchange_learner(arch, dev) for _ in range(2)] for arch in ARCHS}       # two handles per policy


def _seed(arch, k, h):
    return (list(ARCHS).index(arch), k, h)


def _run_exchange(state, rank, world, dev):
    out = {"comm": {}, "calls": [], "blocks": {}, "sms": torch.cuda.get_device_properties(dev).multi_processor_count}
    for arch, hs in state.items():
        out["comm"][arch] = [h["fu"].comm_setup() for h in hs]          # collective; False on every rank if on any
    if not _agree(all(all(v) for v in out["comm"].values())):
        return out
    for hs in state.values():                                           # graph: copy in -> exchange -> copy out
        for h in hs:
            h["x"], h["y"] = torch.empty(h["n"], device=dev), torch.empty_like(h["big"])
            h["graph"] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(h["graph"]):
                h["L"]._bucket.copy_(h["x"])
                h["fu"].allreduce()
                h["y"].copy_(h["big"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for arch, hs in state.items():
        for b, mode in enumerate(MODES):
            ks = range(b * CALLS_PER_BLOCK, (b + 1) * CALLS_PER_BLOCK)
            gs = {(k, hi): I.make_inputs(h["n"], world, _seed(arch, k, hi))[0] for k in ks for hi, h in enumerate(hs)}
            xs = {key: torch.from_numpy(g[rank]).to(dev) for key, g in gs.items()}
            graphed = mode == "graph" or (mode == "mixed" and rank == 0)
            results = []
            torch.cuda.synchronize(dev)
            dist.barrier()
            # ---- block: nothing here asserts
            e0.record()
            for k in ks:
                for hi, h in enumerate(hs):                             # the two handles interleaved, in the same order everywhere
                    if graphed:
                        h["x"].copy_(xs[(k, hi)])
                        h["graph"].replay()
                        results.append((k, hi, h["y"].clone()))
                    else:
                        h["L"]._bucket.copy_(xs[(k, hi)])
                        h["fu"].allreduce()
                        results.append((k, hi, h["big"].clone()))
            e1.record()
            torch.cuda.synchronize(dev)
            # ---- end of block
            out["blocks"][(arch, mode)] = e0.elapsed_time(e1) / len(results)
            for k, hi, got in results:
                n = hs[hi]["n"]
                g = gs[(k, hi)]
                want = I.rank_order_sum(g)
                a = got.cpu().numpy()
                inner = a[PAD:PAD + n].copy()
                outside = np.concatenate([a[:PAD], a[PAD + n:]]).view(np.uint32)
                canon = inner.copy()
                canon[np.isnan(canon)] = np.nan
                out["calls"].append({"arch": arch, "mode": mode, "k": k, "handle": hi, "graphed": graphed,
                                     **I.compare(inner, want), "sentinel_damage": int((outside != I.SENTINEL_BITS).sum()),
                                     "vote": float(inner[n - 1]), "votes": float(g[:, n - 1].sum()),
                                     "digest": hashlib.sha1(canon.tobytes()).hexdigest()})
    # time per exchange, launched back to back on the 3.2 MB bucket (the values are of no interest any more)
    fu = state["bench"][0]["fu"]
    state["bench"][0]["L"]._bucket.zero_()
    torch.cuda.synchronize(dev)
    dist.barrier()
    e0.record()
    for _ in range(16):
        fu.allreduce()
    e1.record()
    torch.cuda.synchronize(dev)
    out["ms_per_exchange"] = e0.elapsed_time(e1) / 16
    return out


@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("world", WORLDS)
def test_exchange_is_the_rank_order_fp32_sum(world, placement, tmp_path, built_lib):
    res = _spawn("exchange", world, placement, tmp_path)
    for r in res:
        assert all(all(v) for v in r["comm"].values()), r["comm"]            # comm_setup: True on every rank
    for arch, (_, n, grid) in ARCHS.items():
        assert n % (4 * world) != 0                                      # the padded tail of publish and collect
        if res[0]["sms"] == 148:
            assert _blocks(n, world, 148) == grid
    expected_calls = len(ARCHS) * len(MODES) * CALLS_PER_BLOCK * 2
    for rank, r in enumerate(res):
        assert len(r["calls"]) == expected_calls
        bad = [c for c in r["calls"] if c["bit_mismatches"] or c["nan_mismatches"] or c["sentinel_damage"]]
        assert not bad, (rank, bad[:4])
        assert all(c["vote"] == c["votes"] for c in r["calls"]), rank
        assert any(c["graphed"] for c in r["calls"]) and any(not c["graphed"] for c in r["calls"])
    # the same bits on every rank (NaN lanes canonicalised)
    for i, c in enumerate(res[0]["calls"]):
        assert all(r["calls"][i]["digest"] == c["digest"] for r in res), c
    print(f"W={world} {placement}: {expected_calls} exchanges per rank bit-identical to the rank-order sum; ms per call by block:",
          {f"{a}/{m}": f"{t:.2f}" for (a, m), t in res[0]["blocks"].items()})
    print(f"  ms per exchange of the 3.2 MB bucket, launched back to back (not a performance number): "
          f"{[round(r['ms_per_exchange'], 3) for r in res]}")


# ---- 3. one data-parallel minibatch through the C ABI against FP64 -------------------------------------------------------------
MB = 1024
MB_CONFIGS = {"clip": {}, "noclip": dict(max_grad_norm=1e9), "vote": {}}


def _setup_minibatch(rank, world, dev):
    from drl_dronenavigation_b200 import ppo
    state = {}
    for cid, over in MB_CONFIGS.items():
        kw = dict(pi_arch=SPEC.pi_arch, vf_arch=SPEC.vf_arch, batch_size=MB, cuda_graph=False, update_impl="fused",
                  target_kl=None, matmul_precision="fp32")
        kw.update(over)
        if cid == "vote":
            kw["target_kl"] = 1e-6 if rank == world - 1 else None      # only the last rank votes
        L = ppo.PPOLearner(13, 4, ppo.PPOConfig(**kw), device=dev)
        g = torch.Generator(device=dev).manual_seed(5)                 # the same non-zero biases on every rank
        with torch.no_grad():
            for p in L.params:
                if p.dim() == 1:
                    p.add_(0.1 * torch.randn(p.shape, device=dev, generator=g))
        ro = R.make_rollout(L.flat_parameters(), SPEC, 2 * MB, seed=300 + 17 * rank, device=dev)
        L.ensure_fused(MB)
        state[cid] = (L, ro)
    return state


def _run_minibatch(state, rank, world, dev):
    out = {"comm": {}, "mb": {}}
    for cid, (L, ro) in state.items():
        fu, cfg = L.fused, L.cfg
        out["comm"][cid] = fu.comm_setup()
        if not _agree(out["comm"][cid]):
            return out
        c = fu.cfg_c
        out["hp"] = dict(lr=c.learning_rate, max_grad_norm=c.max_grad_norm, beta1=c.beta1, beta2=c.beta2, eps=c.adam_eps)
        out["hp_" + cid] = dict(max_grad_norm=c.max_grad_norm, lr=c.learning_rate)
        r = fu.L.dn_ppo_rollout()
        r.obs, r.actions, r.old_log_prob, r.old_values, r.advantages, r.returns = [t.data_ptr() for t in ro]
        gen = torch.Generator(device=dev).manual_seed(17 + rank)
        recs = []
        steps = [(True, k) for k in range(3)] if cid != "vote" else [(True, 0), (False, 1)]
        for begin, k in steps:                       # vote: a second grad + exchange + apply without begin_update
            flat = L.flat_parameters()
            idx = torch.randperm(ro[0].shape[0], device=dev, generator=gen)[:MB]
            margins = R.enforce_margins(flat, SPEC, ro, idx, cfg.clip_range, cfg.clip_range_vf, 1e-3)
            ref = R.minibatch(flat, SPEC, [t[idx] for t in ro], cfg.clip_range, cfg.clip_range_vf, cfg.normalize_advantage,
                              cfg.ent_coef, cfg.vf_coef)
            if begin:
                fu.begin_update()
            fu.minibatch_grad(r, idx)
            torch.cuda.synchronize(dev)
            pre = L._bucket.clone()
            dist.barrier()
            fu.allreduce()
            torch.cuda.synchronize(dev)
            post = L._bucket.clone()
            p0, m0, v0, s0 = fu.params.clone(), fu.exp_avg.clone(), fu.exp_avg_sq.clone(), float(fu.step)
            fu.minibatch_apply()
            st = fu.stats()
            recs.append({"pre": pre.cpu(), "post": post.cpu(), "p0": p0.cpu(), "m0": m0.cpu(), "v0": v0.cpu(), "s0": s0,
                         "p1": fu.params.cpu(), "m1": fu.exp_avg.cpu(), "v1": fu.exp_avg_sq.cpu(), "s1": float(fu.step),
                         "norm": st.last_grad_norm, "steps": st.optimizer_steps, "early_stop": st.early_stop,
                         "ref_grad": ref["grad"].cpu(), "ref_mag": ref["grad_magnitude"].cpu(),
                         "ref_kl": ref["stats"]["approx_kl"], "margins": margins})
        out["mb"][cid] = recs
    return out


@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("world", WORLDS)
def test_data_parallel_minibatch_matches_fp64(world, placement, tmp_path, built_lib):
    res = _spawn("minibatch", world, placement, tmp_path)
    assert all(all(r["comm"].values()) for r in res)
    hp = res[0]["hp"]
    report = {}
    for cid in MB_CONFIGS:
        for k in range(len(res[0]["mb"][cid])):
            recs = [r["mb"][cid][k] for r in res]
            n_params = recs[0]["p0"].numel()
            # the exchange: the rank-order FP32 sum of the ranks' pre-exchange buckets, bit for bit, on every rank
            want = I.rank_order_sum(np.stack([x["pre"].numpy() for x in recs]))
            for rank, x in enumerate(recs):
                cmp = I.compare(x["post"].numpy(), want)
                assert cmp["bit_mismatches"] == 0 and cmp["nan_mismatches"] == 0, (cid, k, rank, cmp)
            post = recs[0]["post"]
            # the summed gradient against the sum of the ranks' FP64 gradients (the bound of test_minibatch_stages_match_fp64)
            gref = sum(x["ref_grad"] for x in recs)
            gmag = sum(x["ref_mag"] for x in recs)
            gerr, floored = R.per_tensor_errors(post[:n_params], gref, SPEC, scale=gmag)
            assert max(gerr.values()) <= 5e-5, (cid, k, gerr)
            report[f"{cid} grad"] = max(report.get(f"{cid} grad", 0.0), max(gerr.values()))
            # the state after apply: bit-identical on every rank
            for x in recs[1:]:
                for key in ("p1", "m1", "v1"):
                    assert torch.equal(x[key], recs[0][key]), (cid, k, key)
                assert x["s1"] == recs[0]["s1"] and x["norm"] == recs[0]["norm"] and x["steps"] == recs[0]["steps"]
            x = recs[0]
            if cid == "vote":
                # only rank W-1 votes: the sum is 1 everywhere, and the apply (and the one after it) changes nothing
                assert recs[-1]["ref_kl"] > 1e3 * 1.5e-6
                for rx in recs:
                    assert float(rx["post"][-1]) == 1.0 and float(rx["pre"][-1]) == (1.0 if rx is recs[-1] else 0.0)
                    assert torch.equal(rx["p1"], rx["p0"]) and torch.equal(rx["m1"], rx["m0"]) and torch.equal(rx["v1"], rx["v0"])
                    assert rx["s1"] == rx["s0"] == 0.0 and rx["steps"] == 0 and rx["early_stop"]
                continue
            assert float(post[-1]) == 0.0 and not x["early_stop"]
            assert x["s0"] == k and x["s1"] == k + 1 and x["steps"] == 1
            # apply divides by world_size: clip_grad_norm_ + Adam in FP64 on the exchanged bucket / W
            p_ref, m_ref, v_ref, norm = R.clip_adam(post[:n_params], x["p0"], x["m0"], x["v0"], x["s0"], lr=hp["lr"],
                                                    max_grad_norm=res[0]["hp_" + cid]["max_grad_norm"], world_size=world,
                                                    beta1=hp["beta1"], beta2=hp["beta2"], eps=hp["eps"])
            aerr = {"param (lr)": float(((x["p1"].double() - p_ref).abs() - R.half_ulp(x["p1"])).max()) / hp["lr"],
                    "exp_avg": R.max_rel(x["m1"], m_ref), "exp_avg_sq": R.max_rel(x["v1"], v_ref),
                    "norm": abs(x["norm"] - norm) / norm}
            assert aerr["param (lr)"] <= 1e-5 and aerr["exp_avg"] <= 1e-5 and aerr["exp_avg_sq"] <= 1e-5, (cid, k, aerr)
            assert aerr["norm"] <= 1e-6, (cid, k, aerr)
            for s, e in aerr.items():
                report[f"{cid} {s}"] = max(report.get(f"{cid} {s}", 0.0), e)
    print(f"W={world} {placement} maxima:", {s: f"{e:.1e}" for s, e in report.items()})


# ---- 4. the learner with real ranks ------------------------------------------------------------------------------------------
B = 4096                            # per rank: 4 minibatches of 1024 per epoch


def _learner(dev, graph, **over):
    from drl_dronenavigation_b200 import ppo
    kw = dict(pi_arch=SPEC.pi_arch, vf_arch=SPEC.vf_arch, batch_size=MB, n_epochs=2, target_kl=None, update_impl="fused",
              cuda_graph=graph, matmul_precision="fp32")
    kw.update(over)
    return ppo.PPOLearner(13, 4, ppo.PPOConfig(**kw), device=dev)


def _flat(L):
    return L.flat_parameters().cpu()


def _counts(L, o):
    return {"impl": L.allreduce_impl, "calls": L.allreduce_calls, **{k: o[k] for k in ("minibatches", "optimizer_steps",
                                                                                      "launched_minibatches", "early_stop")}}


def _setup_learner(rank, world, dev):
    L = _learner(dev, True)
    L.ensure_fused(MB)
    return {"first": L}


def _run_learner(state, rank, world, dev):
    out = {}
    LG = state["first"]
    ro = R.make_rollout(LG.flat_parameters(), SPEC, B, seed=100 + rank, device=dev)
    gen = lambda s: torch.Generator(device=dev).manual_seed(s)          # noqa: E731
    # graph vs launch by launch (the graph holds grad, exchange, apply)
    o = LG.update(*ro, generator=gen(7))
    out["graph"] = {"p": _flat(LG), **_counts(LG, o)}
    LL = _learner(dev, False)
    o = LL.update(*ro, generator=gen(7))
    out["launch"] = {"p": _flat(LL), **_counts(LL, o)}
    # the fallback: two graphs around dist.all_reduce (gloo here); every exchanged bucket recorded
    real = dist.all_reduce
    for name, nccl in (("nccl", True), ("optout", rank == world - 1)):
        if nccl:
            os.environ["DN_PPO_ALLREDUCE"] = "nccl"
        LN = _learner(dev, True)
        seen = []

        def rec(t, *a, **kw):
            if t is LN._bucket:
                pre = t.clone()
                work = real(t, *a, **kw)
                seen.append((pre.cpu(), t.cpu()))
                return work
            return real(t, *a, **kw)
        dist.all_reduce = rec
        try:
            o = LN.update(*ro, generator=gen(7))
        finally:
            dist.all_reduce = real
            os.environ.pop("DN_PPO_ALLREDUCE", None)
        out[name] = {"p": _flat(LN), "exchanges": seen, **_counts(LN, o)}
    # early stop: only the last rank's threshold is in reach (every rank needs a target_kl: the checks sit at the same points)
    # on an on-policy rollout (old log-probs from the policy itself: no vote at the first minibatch)
    for name, graph in (("stop_graph", True), ("stop_launch", False)):
        LE = _learner(dev, graph, n_epochs=5, learning_rate=1e-2, target_kl=1e-3 if rank == world - 1 else 1e9)
        g = gen(200 + rank)
        obs = torch.randn(B, 13, device=dev, generator=g)
        a, logp, v = LE.act(obs, generator=g)
        adv, ret = torch.randn(B, device=dev, generator=g), v + torch.randn(B, device=dev, generator=g)
        o = LE.update(obs, a, logp, v, adv, ret, generator=gen(9))
        out[name] = {"p": _flat(LE), **_counts(LE, o)}
    # handle re-creation: a forward on more rows than max_rows re-creates the handle; the next update sets up the exchange again
    for name, L in (("recreate_graph", LG), ("recreate_launch", LL)):
        old = L.fused
        L.forward(ro[0][:MB + 256])
        fu = L.fused
        o = L.update(*ro, generator=gen(8))
        out[name] = {"p": _flat(L), "new_handle": fu is not old and fu.max_rows == MB + 256, "comm_ready": fu.comm_ready,
                     **_counts(L, o)}
    return out


_SETUP = {"exchange": _setup_exchange, "minibatch": _setup_minibatch, "learner": _setup_learner}
_RUN = {"exchange": _run_exchange, "minibatch": _run_minibatch, "learner": _run_learner}


@pytest.fixture(scope="module", params=[(w, p) for w in WORLDS for p in PLACEMENTS], ids=lambda x: f"{x[0]}-{x[1]}")
def learner_runs(request, built_lib, tmp_path_factory):
    world, placement = request.param
    return world, _spawn("learner", world, placement, tmp_path_factory.mktemp(f"learner{world}{placement}"))


def _same_everywhere(res, case, key="p"):
    for rank, r in enumerate(res[1:], start=1):
        assert torch.equal(r[case][key], res[0][case][key]), (case, rank)


def test_graph_and_launch_by_launch_agree_bit_for_bit(learner_runs):
    world, res = learner_runs
    for r in res:
        for case in ("graph", "launch"):
            c = r[case]
            assert c["impl"] == "peer" and c["calls"] == c["minibatches"] == c["optimizer_steps"] == c["launched_minibatches"] == 8
        assert torch.equal(r["graph"]["p"], r["launch"]["p"])
    _same_everywhere(res, "graph")


def test_fallback_path_agrees_with_the_rank_order_sum(learner_runs):
    world, res = learner_runs
    for r in res:
        c = r["nccl"]
        assert c["impl"] == "nccl" and c["calls"] == c["minibatches"] == 8 and len(c["exchanges"]) == 8
    _same_everywhere(res, "nccl")
    worst = 0.0
    for j in range(8):
        pre = np.stack([r["nccl"]["exchanges"][j][0].numpy() for r in res])
        want = I.rank_order_sum(pre)
        bound = (world - 1) * 2.0 ** -23 * np.abs(pre.astype(np.float64)).sum(0)
        for r in res:
            got = r["nccl"]["exchanges"][j][1].numpy()
            if world == 2:                       # a sum of two terms does not depend on the order
                assert I.compare(got, want)["bit_mismatches"] == 0, j
            err = np.abs(got.astype(np.float64) - want)
            assert np.all(err <= bound), (j, float((err - bound).max()))
            worst = max(worst, float((err / np.maximum(bound, 1e-300)).max()))
    if world == 2:
        for r in res:
            assert torch.equal(r["nccl"]["p"], r["graph"]["p"])
    print(f"W={world}: fallback exchange vs rank-order sum, max error / ((W-1) ulp of the magnitude sum) = {worst:.2f}")


def test_one_rank_opting_out_sends_every_rank_to_the_fallback(learner_runs):
    world, res = learner_runs
    for r in res:
        assert r["optout"]["impl"] == "nccl" and r["optout"]["calls"] == 8
        assert torch.equal(r["optout"]["p"], r["nccl"]["p"])
    _same_everywhere(res, "optout")


def test_early_stop_is_taken_together(learner_runs):
    world, res = learner_runs
    keys = ("minibatches", "optimizer_steps", "launched_minibatches", "calls", "early_stop")
    for case in ("stop_graph", "stop_launch"):
        c0 = res[0][case]
        assert c0["early_stop"] and c0["minibatches"] == c0["optimizer_steps"] + 1 and c0["minibatches"] >= 2, c0
        assert c0["calls"] == c0["launched_minibatches"] and c0["impl"] == "peer"
        for r in res:
            assert {k: r[case][k] for k in keys} == {k: c0[k] for k in keys}
        _same_everywhere(res, case)
    for r in res:
        assert torch.equal(r["stop_graph"]["p"], r["stop_launch"]["p"])
        assert {k: r["stop_graph"][k] for k in keys} == {k: r["stop_launch"][k] for k in keys}
    print(f"W={world}: early stop after {res[0]['stop_graph']['minibatches']} minibatches, "
          f"{res[0]['stop_graph']['launched_minibatches']} launched")


def test_recreated_handle_sets_up_the_exchange_again(learner_runs):
    world, res = learner_runs
    for r in res:
        for case in ("recreate_graph", "recreate_launch"):
            c = r[case]
            assert c["new_handle"] and c["comm_ready"] and c["impl"] == "peer" and c["calls"] == 16 and c["minibatches"] == 8
        assert torch.equal(r["recreate_graph"]["p"], r["recreate_launch"]["p"])
        assert not torch.equal(r["recreate_graph"]["p"], r["graph"]["p"])
    _same_everywhere(res, "recreate_graph")
