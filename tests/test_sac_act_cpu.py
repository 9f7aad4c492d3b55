"""dn_sac_act without a GPU: the numpy restatement of its draw layout (tests/sac_act_reference.py) against the PPO sampler's
words and sac.py::Actor in FP64, the statistics of its normals and uniforms, the tag in header / binding / restatement, the
argument checks of dn_sac_act and dn_sac_actor_create, the ctypes layouts, FusedSACActor.shapes_ok against the library,
and SACConfig.rollout_impl."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

from tests.conftest import ROOT
from tests import ppo_act_reference as P
from tests import sac_act_reference as R

DN_EINVAL = -1


def test_tag_is_the_same_in_header_binding_and_restatement_and_differs_from_the_other_streams():
    text = open(os.path.join(ROOT, "include", "dnsac.h")).read()
    tag = int(re.search(r"#define DN_SAC_ACT_TAG (0x[0-9A-Fa-f]+)u", text).group(1), 16)
    from drl_dronenavigation_b200 import _lib
    assert tag == _lib.DN_SAC_ACT_TAG == R.DN_SAC_ACT_TAG == int.from_bytes(b"SACA", "big")
    assert tag not in (0, 1, P.DN_PPO_ACT_TAG)    # spawn draws use 0 and 1; dn_ppo_act its own tag


def test_with_the_ppo_tag_the_words_are_the_ppo_samplers():
    rng = np.random.default_rng(3)
    for _ in range(20):
        seed, counter = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 2 ** 32))
        rows = rng.integers(0, 2 ** 40, size=64)
        np.testing.assert_array_equal(R.philox_words(seed, counter, rows, tag=P.DN_PPO_ACT_TAG), P.philox_words(seed, counter, rows))
        assert not np.array_equal(R.philox_words(seed, counter, rows), P.philox_words(seed, counter, rows))


def test_the_words_match_the_oracle_generator():
    from oracle.dyn_oracle import philox4x32_10
    for seed, counter, row in ((42, 0, 0), (7, 3, (1 << 33) + 9), (0xFEDCBA9876543210, 0xFFFFFFFF, 12345)):
        want = philox4x32_10((counter & 0xFFFFFFFF, R.DN_SAC_ACT_TAG, row & 0xFFFFFFFF, row >> 32), (seed & 0xFFFFFFFF, seed >> 32))
        assert [int(w) for w in R.philox_words(seed, counter, [row])[0]] == list(want)


def test_the_squashed_gaussian_equals_the_torch_actor_in_fp64():
    from drl_dronenavigation_b200.sac import Actor
    torch.manual_seed(0)
    for arch, act_dim in (((256, 256), 4), ((128,), 1), ((128, 256, 128, 384), 3)):
        actor = Actor(13, act_dim, arch).double()
        with torch.no_grad():
            actor.log_std.bias.fill_(-0.5)
        obs = torch.randn(300, 13, dtype=torch.float64) * 3
        eps = R.normals(5, 2, np.arange(300), act_dim)
        a_t, lp_t = actor(obs, eps=torch.from_numpy(eps))
        params = {k: v.numpy() for k, v in actor.state_dict().items()}
        _, mu, ls, a, lp = R.actor_forward(params, obs.numpy(), eps)
        np.testing.assert_allclose(a, a_t.detach().numpy(), rtol=0, atol=1e-12)
        np.testing.assert_allclose(lp, lp_t.detach().numpy(), rtol=1e-12, atol=1e-9)
        a_d, _ = actor(obs, deterministic=True)
        np.testing.assert_allclose(R.actor_forward(params, obs.numpy())[3], a_d.detach().numpy(), rtol=0, atol=1e-12)


def test_a_million_normals_pass_ks_and_uniform_mode_is_uniform_on_minus_one_one():
    from scipy import stats
    rows = np.arange(1 << 18)
    z = np.concatenate([R.normals(99, c, rows, 4) for c in range(4)])          # [2^20, 4]
    assert z.shape[0] >= 10 ** 6
    for a in range(4):
        assert stats.kstest(z[:, a], "norm").pvalue > 0.01, a
    u = np.concatenate([R.uniform_actions(99, c, rows, 4) for c in range(4)])
    assert u.dtype == np.float32 and u.min() >= -1.0 and u.max() < 1.0
    for a in range(4):
        assert stats.kstest(u[:, a].astype(np.float64), "uniform", args=(-1.0, 2.0)).pvalue > 0.01, a
    # every value is a multiple of 2^-23 in [-1, 1): the 24-bit uniforms map exactly
    assert np.all(np.mod(u.astype(np.float64) + 1.0, 2.0 ** -23) == 0.0)


def test_draws_depend_on_the_global_row_id_only():
    n = 1000
    both = R.philox_words(9, 3, np.arange(2 * n))
    np.testing.assert_array_equal(both[n:], R.philox_words(9, 3, n + np.arange(n)))
    assert not np.array_equal(R.philox_words(9, 3, np.arange(n)), R.philox_words(9, 4, np.arange(n)))
    assert not np.array_equal(R.philox_words(9, 3, np.arange(n)), R.philox_words(10, 3, np.arange(n)))


def test_struct_layouts_match_the_header(built_lib):
    from drl_dronenavigation_b200 import _lib
    assert C.sizeof(_lib.dn_sac_sample) == 8 + 8 + 8 + 4 + 4
    assert [f for f, _ in _lib.dn_sac_sample._fields_] == ["seed", "row_id_offset", "counter", "mode", "reserved0"]
    assert C.sizeof(_lib.dn_sac_actor_config) == 10 * 4 + (2 * 4 + 5) * 8
    assert _lib.dn_sac_actor_config.w_off.offset == 40
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dnsac.h")).read(), flags=re.S)
    assert set(re.findall(r"\b(dn_[a-z_]+)\s*\(", text)) == set(_lib.SAC_SYMBOLS)
    for n in _lib.SAC_SYMBOLS:
        assert hasattr(built_lib, n)


def test_dn_sac_act_rejects_bad_arguments_without_a_gpu(built_lib):
    """Every argument is checked before the handle is read: a stand-in handle (a host buffer) is never dereferenced."""
    from drl_dronenavigation_b200 import _lib
    buf = (C.c_float * 64)()
    fake = C.cast(buf, C.c_void_p)
    ctr = (C.c_int64 * 1)()

    def sample(**kw):
        s = _lib.dn_sac_sample()
        s.seed, s.row_id_offset, s.counter, s.mode = 1, 0, C.cast(ctr, C.c_void_p), _lib.DN_SAC_SAMPLE
        for k, v in kw.items():
            setattr(s, k, v)
        return s
    ok = sample()
    cases = [
        ((None, buf, 4, C.byref(ok), buf, buf, None), b"null"),
        ((fake, None, 4, C.byref(ok), buf, buf, None), b"null"),
        ((fake, buf, 4, None, buf, buf, None), b"null"),
        ((fake, buf, 4, C.byref(ok), None, buf, None), b"null"),
        ((fake, buf, 4, C.byref(sample(counter=None)), buf, buf, None), b"counter"),
        ((fake, buf, 4, C.byref(sample(counter=None, mode=_lib.DN_SAC_UNIFORM)), buf, buf, None), b"counter"),
        ((fake, buf, 4, C.byref(sample(mode=3)), buf, buf, None), b"mode"),
        ((fake, buf, 4, C.byref(sample(mode=-1)), buf, buf, None), b"mode"),
        ((fake, buf, 4, C.byref(sample(row_id_offset=-1)), buf, buf, None), b"row_id_offset"),
        ((fake, buf, 0, C.byref(ok), buf, buf, None), b"rows"),
        ((fake, buf, -5, C.byref(ok), buf, None, None), b"rows"),
    ]
    for args, word in cases:
        assert built_lib.dn_sac_act(*args) == DN_EINVAL
        msg = built_lib.dn_last_error()
        assert b"dn_sac_act" in msg and word in msg, (args, msg)


def _config(arch, obs_dim=13, act_dim=4, max_rows=256):
    from drl_dronenavigation_b200 import _lib
    c = _lib.dn_sac_actor_config()
    c.abi_version, c.obs_dim, c.act_dim, c.max_rows, c.precision = _lib.DN_ABI_VERSION, obs_dim, act_dim, max_rows, _lib.DN_MLP_BF16X3
    c.n_hidden = len(arch)
    off, prev = 0, obs_dim
    for l, w in enumerate(arch[:_lib.DN_SAC_MAX_LAYERS]):
        c.hidden[l] = w
        c.w_off[l], c.b_off[l] = off, off + w * prev
        off += w * prev + w
        prev = w
    last = arch[-1] if arch else 128
    c.mu_w_off, c.mu_b_off = off, off + act_dim * last
    off += act_dim * last + act_dim
    c.log_std_w_off, c.log_std_b_off = off, off + act_dim * last
    c.n_params = off + act_dim * last + act_dim
    return c


def _create_error(c):
    buf = (C.c_float * 8)()
    h = C.c_void_p()
    from drl_dronenavigation_b200 import _lib
    rc = _lib.lib().dn_sac_actor_create(C.byref(c), 0, C.cast(buf, C.c_void_p), C.byref(h))
    assert rc < 0 and not h.value          # no device here: a valid config fails only at the device lookup
    msg = _lib.lib().dn_last_error()
    return None if b"no CUDA device" in msg or b"sm_100a" in msg or b"device index" in msg else msg


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the config validation on a machine without a device")
def test_dn_sac_actor_create_validates_the_config_before_touching_a_device(built_lib):
    from drl_dronenavigation_b200 import _lib
    assert _create_error(_config((256, 256))) is None
    bad = []
    for field, value, word in (("abi_version", 999, b"abi_version"), ("obs_dim", 0, b"obs_dim"), ("obs_dim", 65, b"obs_dim"),
                               ("act_dim", 0, b"act_dim"), ("act_dim", 5, b"act_dim"), ("max_rows", 100, b"max_rows"),
                               ("max_rows", 0, b"max_rows"), ("precision", 7, b"precision"), ("n_params", 10, b"n_params"),
                               ("mu_w_off", -1, b"n_params")):
        c = _config((256, 256))
        setattr(c, field, value)
        bad.append((field, value, word, _create_error(c)))
    c = _config((256, 256))
    c.log_std_b_off = c.n_params - 1                  # the last tensor runs past the end
    bad.append(("log_std_b_off", "end", b"n_params", _create_error(c)))
    for field, value, word, msg in bad:
        assert msg is not None and b"dn_sac_actor_create" in msg and word in msg, (field, value, msg)
    assert built_lib.dn_sac_actor_create(None, 0, None, None) == DN_EINVAL


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the config validation on a machine without a device")
def test_shapes_ok_agrees_with_dn_sac_actor_create(built_lib):
    from drl_dronenavigation_b200.sac import FusedSACActor
    widths = (64, 128, 192, 256, 384, 512, 640, 1024)
    archs = [()] + [(w,) for w in widths] + [(w, 256) for w in widths] + [(256, w, 128) for w in widths] + \
        [(128, 128, 128, w) for w in widths] + [(128,) * 5, (256,) * 4, (512,) * 4]
    n = 0
    for arch in archs:
        for obs_dim in (0, 1, 12, 13, 64, 65):
            for act_dim in (0, 1, 2, 3, 4, 5):
                want = FusedSACActor.shapes_ok(arch, obs_dim, act_dim)
                c = _config(arch if arch else (128,), obs_dim, act_dim)
                if not arch:
                    c.n_hidden = 0
                elif len(arch) > 4:
                    c.n_hidden = len(arch)
                assert (_create_error(c) is None) == want, (arch, obs_dim, act_dim)
                n += 1
    assert n > 1000


def test_rollout_impl_validation():
    from drl_dronenavigation_b200.argparser import parse_args
    from drl_dronenavigation_b200.sac import SACConfig, SACLearner
    assert SACConfig().rollout_impl == "torch"
    assert parse_args(["--agent", "SAC", "--rollout_impl", "fused"]).rollout_impl == "fused"
    with pytest.raises(ValueError, match="rollout_impl"):
        SACConfig(rollout_impl="graph")
    with pytest.raises(RuntimeError, match="compute-capability-10"):
        SACLearner(13, 4, SACConfig(rollout_impl="fused"), device="cpu")
    with pytest.raises(RuntimeError, match="compute-capability-10"):
        SACLearner(13, 4, SACConfig(rollout_impl="fused", pi_arch=(100,)), device="cpu")
    SACLearner(13, 4, SACConfig(), device="cpu")            # the default builds as before


def test_fused_learner_parameters_start_equal_to_the_torch_learners(monkeypatch):
    """The flat vector re-seats the actor's Parameters without changing a bit (checked on the CPU by skipping the device check)."""
    from drl_dronenavigation_b200 import sac
    monkeypatch.setattr(sac.FusedSACActor, "check_supported", staticmethod(lambda *a: None))
    ref = sac.SACLearner(13, 4, sac.SACConfig(), device="cpu")
    fused = sac.SACLearner(13, 4, sac.SACConfig(rollout_impl="fused"), device="cpu")
    for (k, a), (k2, b) in zip(ref.actor.state_dict().items(), fused.actor.state_dict().items()):
        assert k == k2 and torch.equal(a, b)
    for a, b in zip(ref.critic.parameters(), fused.critic.parameters()):
        assert torch.equal(a, b)
    flat, off = fused.actor_flat, 0
    for p in fused.actor.parameters():
        assert p.data_ptr() == flat.data_ptr() + 4 * off
        off += p.numel()
    assert off == flat.numel()
    assert math.isfinite(float(flat.abs().sum()))
