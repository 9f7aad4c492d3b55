"""numpy / FP64 restatement of dn_sac_act (include/dnsac.h, "Draw layout"): the Philox words of every row for a given tag,
the Box-Muller normals, the uniform actions of DN_SAC_UNIFORM, and SB3's squashed-Gaussian actor (sac.py::Actor.forward)
evaluated in float64 on given weights and noise."""
import math

import numpy as np

DN_SAC_ACT_TAG = 0x53414341          # include/dnsac.h ("SACA")
LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0

_MASK = np.uint64(0xFFFFFFFF)


def philox_words(seed: int, counter: int, row_ids, tag: int = DN_SAC_ACT_TAG) -> np.ndarray:
    """[n, 4] uint32: Philox4x32-10 with key (seed lo, seed hi), counter (counter mod 2^32, tag, row lo, row hi)."""
    rid = np.asarray(row_ids, dtype=np.uint64).reshape(-1)
    c0 = np.full(rid.shape, int(counter) & 0xFFFFFFFF, dtype=np.uint64)
    c1 = np.full(rid.shape, int(tag) & 0xFFFFFFFF, dtype=np.uint64)
    c2, c3 = rid & _MASK, rid >> np.uint64(32)
    k0, k1 = np.uint64(int(seed) & 0xFFFFFFFF), np.uint64((int(seed) >> 32) & 0xFFFFFFFF)
    m0, m1, w0, w1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                      # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + w0) & _MASK, (k1 + w1) & _MASK
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def u01(w):
    return (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24          # [0, 1)


def u01_open(w):
    return ((np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24  # (0, 1]


def normals(seed: int, counter: int, row_ids, act_dim: int = 4) -> np.ndarray:
    """[n, act_dim] FP64 eps of DN_SAC_SAMPLE: Box-Muller on (x, y) and (z, w)."""
    w = philox_words(seed, counter, row_ids)
    r1, r2 = np.sqrt(-2.0 * np.log(u01_open(w[:, 0]))), np.sqrt(-2.0 * np.log(u01_open(w[:, 2])))
    t1, t2 = 2.0 * np.pi * u01(w[:, 1]), 2.0 * np.pi * u01(w[:, 3])
    return np.stack([r1 * np.cos(t1), r1 * np.sin(t1), r2 * np.cos(t2), r2 * np.sin(t2)], axis=-1)[:, :act_dim]


def uniform_actions(seed: int, counter: int, row_ids, act_dim: int = 4) -> np.ndarray:
    """[n, act_dim] float32 actions of DN_SAC_UNIFORM: 2 u01(word a) - 1 (exact in FP32)."""
    return (2.0 * u01(philox_words(seed, counter, row_ids)[:, :act_dim]) - 1.0).astype(np.float32)


def squash(mu, log_std, eps=None):
    """SquashedDiagGaussian in FP64: (action, log_prob).  eps None: deterministic (action = tanh(mu), log_prob with eps = 0)."""
    mu, ls = np.asarray(mu, np.float64), np.asarray(log_std, np.float64)
    eps = np.zeros_like(mu) if eps is None else np.asarray(eps, np.float64)
    a = np.tanh(mu + np.exp(ls) * eps)
    logp = (-0.5 * eps ** 2 - ls - 0.5 * math.log(2.0 * math.pi)).sum(-1) - np.log(1.0 - a ** 2 + 1e-6).sum(-1)
    return a, logp


def actor_forward(params, obs, eps=None):
    """sac.py::Actor.forward in FP64.  params: dict of numpy arrays (state-dict names of Actor); returns hidden activations
    [h1, ..], mu, log_std (clamped), action, log_prob."""
    h = np.asarray(obs, np.float64)
    hs = []
    l = 0
    while f"latent.{2 * l}.weight" in params:
        h = np.maximum(h @ np.asarray(params[f"latent.{2 * l}.weight"], np.float64).T + np.asarray(params[f"latent.{2 * l}.bias"], np.float64), 0.0)
        hs.append(h)
        l += 1
    mu = h @ np.asarray(params["mu.weight"], np.float64).T + np.asarray(params["mu.bias"], np.float64)
    ls = np.clip(h @ np.asarray(params["log_std.weight"], np.float64).T + np.asarray(params["log_std.bias"], np.float64), LOG_STD_MIN, LOG_STD_MAX)
    a, logp = squash(mu, ls, eps)
    return hs, mu, ls, a, logp
