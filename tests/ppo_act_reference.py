"""numpy / FP64 restatement of dn_ppo_act's sampler (include/dnppo.h, "Draw layout"): the Philox words of every row,
the Box-Muller normals and the Gaussian log-prob.  The scalar generator is oracle.dyn_oracle.philox4x32_10; `philox_words`
is the same function vectorised over rows (checked against it in tests/test_ppo_act_sampler_cpu.py)."""
import math

import numpy as np

DN_PPO_ACT_TAG = 0x50504F41          # include/dnppo.h
Z_MAX = math.sqrt(48.0 * math.log(2.0))   # |z| bound of 24-bit uniforms: sqrt(-2 ln 2^-24)

_MASK = np.uint64(0xFFFFFFFF)


def philox_words(seed: int, counter: int, row_ids) -> np.ndarray:
    """[n, 4] uint32: Philox4x32-10 with key (seed lo, seed hi), counter (counter mod 2^32, DN_PPO_ACT_TAG, row lo, row hi)."""
    rid = np.asarray(row_ids, dtype=np.uint64).reshape(-1)
    c0 = np.full(rid.shape, int(counter) & 0xFFFFFFFF, dtype=np.uint64)
    c1 = np.full(rid.shape, DN_PPO_ACT_TAG, dtype=np.uint64)
    c2, c3 = rid & _MASK, rid >> np.uint64(32)
    k0, k1 = np.uint64(int(seed) & 0xFFFFFFFF), np.uint64((int(seed) >> 32) & 0xFFFFFFFF)
    m0, m1, w0, w1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                      # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + w0) & _MASK, (k1 + w1) & _MASK
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def u01(w):
    return (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24          # [0, 1), exact in FP32 too


def u01_open(w):
    return ((np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24  # (0, 1]


def normals(seed: int, counter: int, row_ids, act_dim: int = 4) -> np.ndarray:
    """[n, act_dim] FP64 z of the rows: Box-Muller on (x, y) and (z, w)."""
    w = philox_words(seed, counter, row_ids)
    r1, r2 = np.sqrt(-2.0 * np.log(u01_open(w[:, 0]))), np.sqrt(-2.0 * np.log(u01_open(w[:, 2])))
    t1, t2 = 2.0 * np.pi * u01(w[:, 1]), 2.0 * np.pi * u01(w[:, 3])
    z = np.stack([r1 * np.cos(t1), r1 * np.sin(t1), r2 * np.cos(t2), r2 * np.sin(t2)], axis=-1)
    return z[:, :act_dim]


def log_prob(action, mean, log_std) -> np.ndarray:
    """FP64 diagonal-Gaussian log-density of `action` (rows) under N(mean, exp(log_std)^2)."""
    a, m, ls = (np.asarray(v, dtype=np.float64) for v in (action, mean, log_std))
    d = a - m
    return (-0.5 * d * d * np.exp(-2.0 * ls) - ls - 0.5 * math.log(2.0 * math.pi)).sum(-1)
