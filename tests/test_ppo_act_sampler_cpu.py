"""dn_ppo_act without a GPU: the numpy restatement of its draw layout (tests/ppo_act_reference.py) against the oracle's Philox
and known-answer words, the statistics of the normals it yields, the header / binding constants, the argument checks of
the C entry point, and the Python switches (PPOConfig.rollout_impl, --rollout_impl)."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from tests.conftest import ROOT
from tests import ppo_act_reference as R

# (seed, counter, global row id) -> the four Philox words of the row (pinned: any change of the layout changes them)
KAT = [
    ((42, 0, 0), (0x502F3D74, 0x2718DED2, 0xE45E9C19, 0xA9CA9B5D)),
    ((42, 1, 0), (0x08F273FA, 0x5FFAFF4D, 0xF03B42EF, 0x551D08D3)),
    ((42, 0, 1), (0xA75796FD, 0xF9B27B95, 0xD8868500, 0x69FD616B)),
    ((0x123456789ABCDEF0, 7, (1 << 32) + 5), (0x090F0B82, 0x38581506, 0xE16564EC, 0xC2E34BD6)),
    ((1, 0xFFFFFFFF, 65535), (0x67A0702A, 0x5C6D7BB6, 0x5D68B98A, 0x545C6BBE)),
]


def test_tag_is_the_same_in_header_binding_and_restatement_and_differs_from_the_spawn_blocks():
    text = open(os.path.join(ROOT, "include", "dnppo.h")).read()
    tag = int(re.search(r"#define DN_PPO_ACT_TAG (0x[0-9A-Fa-f]+)u", text).group(1), 16)
    from drl_dronenavigation_b200 import _lib
    assert tag == _lib.DN_PPO_ACT_TAG == R.DN_PPO_ACT_TAG
    assert tag not in (0, 1)          # the random-spawn draws use 0 and 1 in the second counter word


@pytest.mark.parametrize("key,words", KAT)
def test_restatement_reproduces_the_known_answer_words(key, words):
    from oracle.dyn_oracle import philox4x32_10
    seed, counter, row = key
    assert tuple(int(w) for w in R.philox_words(seed, counter, [row])[0]) == words
    # the same words from the oracle's scalar Philox with the documented counter / key layout
    assert tuple(philox4x32_10((counter & 0xFFFFFFFF, R.DN_PPO_ACT_TAG, row & 0xFFFFFFFF, row >> 32),
                               (seed & 0xFFFFFFFF, seed >> 32))) == words


def test_vectorised_philox_matches_the_oracle_on_random_points():
    from oracle.dyn_oracle import philox4x32_10
    rng = np.random.default_rng(5)
    for _ in range(40):
        seed, counter = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 2 ** 32))
        rows = rng.integers(0, 2 ** 40, size=3)
        got = R.philox_words(seed, counter, rows)
        for r, w in zip(rows, got):
            r = int(r)
            assert [int(v) for v in w] == philox4x32_10((counter, R.DN_PPO_ACT_TAG, r & 0xFFFFFFFF, r >> 32), (seed & 0xFFFFFFFF, seed >> 32))


def test_box_muller_mapping_of_the_known_answer_words():
    (seed, counter, row), (x, y, z, w) = KAT[0]
    u = lambda v: (v >> 8) * 2.0 ** -24
    uo = lambda v: ((v >> 8) + 1) * 2.0 ** -24
    r1, r2 = math.sqrt(-2 * math.log(uo(x))), math.sqrt(-2 * math.log(uo(z)))
    want = [r1 * math.cos(2 * math.pi * u(y)), r1 * math.sin(2 * math.pi * u(y)), r2 * math.cos(2 * math.pi * u(w)), r2 * math.sin(2 * math.pi * u(w))]
    np.testing.assert_allclose(R.normals(seed, counter, [row], 4)[0], want, rtol=0, atol=1e-15)
    np.testing.assert_array_equal(R.normals(seed, counter, [row], 3)[0], R.normals(seed, counter, [row], 4)[0, :3])
    np.testing.assert_array_equal(R.normals(seed, counter, [row], 1)[0], R.normals(seed, counter, [row], 4)[0, :1])


def test_normals_are_bounded_as_documented():
    assert abs(R.Z_MAX - 5.768) < 1e-3
    extreme = np.sqrt(-2.0 * np.log(R.u01_open(np.array([0], dtype=np.uint32))))[0]   # smallest u01_open = 2^-24
    assert extreme == pytest.approx(R.Z_MAX, rel=1e-12)


def test_a_million_draws_are_standard_normal_and_uncorrelated():
    """10^6 rows x 4 components (4 counters x 2^18 rows, seed fixed: the statistics below are deterministic)."""
    from scipy import stats
    rows = np.arange(1 << 18)
    zs = [R.normals(1234, c, rows, 4) for c in range(5)]
    z = np.concatenate(zs[:4])                           # [2^20, 4]
    assert z.shape[0] >= 10 ** 6
    assert np.abs(z).max() <= R.Z_MAX
    for a in range(4):
        ks = stats.kstest(z[:, a], "norm")
        assert ks.pvalue > 0.01, (a, ks)
        assert abs(z[:, a].mean()) < 5e-3 and abs(z[:, a].std() - 1.0) < 5e-3
    c = np.corrcoef(z.T)
    off = np.abs(c - np.eye(4)).max()
    assert off < 5e-3, c
    # consecutive counters of the same row, and neighbouring rows of the same counter
    for k in range(4):
        for a in range(4):
            assert abs(np.corrcoef(zs[k][:, a], zs[k + 1][:, a])[0, 1]) < 5e-3
            assert abs(np.corrcoef(zs[k][:-1, a], zs[k][1:, a])[0, 1]) < 5e-3


def test_draws_depend_on_the_global_row_id_only():
    """Shard invariance of the layout: rows [N, 2N) of one call are rows [0, N) of a call whose offset is N."""
    n = 1000
    both = R.philox_words(9, 3, np.arange(2 * n))
    np.testing.assert_array_equal(both[n:], R.philox_words(9, 3, n + np.arange(n)))
    assert not np.array_equal(R.philox_words(9, 3, np.arange(n)), R.philox_words(9, 4, np.arange(n)))
    assert not np.array_equal(R.philox_words(9, 3, np.arange(n)), R.philox_words(10, 3, np.arange(n)))


def test_sample_struct_layout(built_lib):
    from drl_dronenavigation_b200 import _lib
    assert C.sizeof(_lib.dn_ppo_sample) == 8 + 8 + 8 + 4 + 4 + 4 + 4          # + tail padding to 8
    assert [f for f, _ in _lib.dn_ppo_sample._fields_] == ["seed", "row_id_offset", "counter", "deterministic", "low", "high"]


def test_dn_ppo_act_rejects_bad_arguments_without_a_gpu(built_lib):
    """Every argument is checked before the handle is read: a stand-in handle (a host buffer) is never dereferenced."""
    from drl_dronenavigation_b200 import _lib
    DN_EINVAL = -1
    buf = (C.c_float * 64)()
    fake = C.cast(buf, C.c_void_p)
    ctr = (C.c_int64 * 1)()

    def sample(**kw):
        s = _lib.dn_ppo_sample()
        s.seed, s.row_id_offset, s.counter, s.deterministic, s.low, s.high = 1, 0, C.cast(ctr, C.c_void_p), 0, -1.0, 1.0
        for k, v in kw.items():
            setattr(s, k, v)
        return s
    ok = sample()
    cases = [
        ((None, buf, 4, C.byref(ok), buf, buf, buf, buf, None), b"null"),
        ((fake, None, 4, C.byref(ok), buf, buf, buf, buf, None), b"null"),
        ((fake, buf, 4, None, buf, buf, buf, buf, None), b"null"),
        ((fake, buf, 4, C.byref(ok), None, buf, buf, buf, None), b"null"),
        ((fake, buf, 4, C.byref(ok), buf, buf, None, buf, None), b"null"),
        ((fake, buf, 4, C.byref(ok), buf, buf, buf, None, None), b"null"),
        ((fake, buf, 4, C.byref(sample(counter=None)), buf, buf, buf, buf, None), b"counter"),
        ((fake, buf, 4, C.byref(sample(deterministic=2)), buf, buf, buf, buf, None), b"deterministic"),
        ((fake, buf, 4, C.byref(sample(row_id_offset=-1)), buf, buf, buf, buf, None), b"row_id_offset"),
        ((fake, buf, 4, C.byref(sample(low=1.0, high=-1.0)), buf, buf, buf, buf, None), b"low"),
        ((fake, buf, 4, C.byref(sample(low=float("nan"))), buf, buf, buf, buf, None), b"low"),
        ((fake, buf, 0, C.byref(ok), buf, buf, buf, buf, None), b"rows"),
        ((fake, buf, -5, C.byref(ok), buf, buf, buf, buf, None), b"rows"),
    ]
    for args, word in cases:
        assert built_lib.dn_ppo_act(*args) == DN_EINVAL
        msg = built_lib.dn_last_error()
        assert b"dn_ppo_act" in msg and word in msg, (args, msg)


def test_rollout_impl_switches():
    from drl_dronenavigation_b200.argparser import parse_args
    from drl_dronenavigation_b200.ppo import PPOConfig
    assert PPOConfig().rollout_impl == "torch"                       # the default rollout (and its noise) is unchanged
    assert parse_args([]).rollout_impl == "torch"
    assert parse_args(["--rollout_impl", "fused"]).rollout_impl == "fused"
    with pytest.raises(SystemExit):
        parse_args(["--rollout_impl", "triton"])


class _CpuEnv:
    """The attributes PPOTrainer reads from an env, on the CPU (no fused handle can exist there)."""
    device, num_envs, obs_dim, env_id_offset = "cpu", 8, 13, 0

    def reset(self):
        import torch
        return torch.zeros(self.num_envs, self.obs_dim)


def test_fused_rollout_without_the_fused_handle_raises():
    from drl_dronenavigation_b200.ppo import PPOConfig, PPOTrainer
    small = dict(pi_arch=(128,), vf_arch=(128,), batch_size=8, n_steps=4)
    with pytest.raises(RuntimeError, match="rollout_impl='fused' needs the fused PPO handle"):
        PPOTrainer(_CpuEnv(), PPOConfig(rollout_impl="fused", **small), rollout_steps=4)
    with pytest.raises(ValueError, match="rollout_impl"):
        PPOTrainer(_CpuEnv(), PPOConfig(rollout_impl="graph", **small), rollout_steps=4)
    PPOTrainer(_CpuEnv(), PPOConfig(**small), rollout_steps=4)        # the default builds as before
