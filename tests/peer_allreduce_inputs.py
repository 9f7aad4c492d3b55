"""Inputs of the gradient all-reduce tests and their exact rank-order FP32 sum.

``make_inputs(n, world, seed)`` builds the buckets of ALL ranks for one call of ``dn_ppo_allreduce`` (include/dnppo.h), so every
rank (and the test's parent process) can rebuild every rank's input and the expected result from the seed alone.  Element
n - 1 is each rank's 0/1 early-stop vote; the other lanes fall into these categories:

  * wide: independent random values over the scales 2^-20 .. 2^20;
  * order: lanes whose rank-order sum ((g0 + g1) + g2) + ... differs in FP32 from the reversed order and from a pairwise tree
    (W >= 3; with two ranks every order gives the same sum), so a kernel that summed in another order would not match;
  * neg_zero (every rank -0: the sum is -0), mixed_zero (-0 and +0: the sum is +0);
  * subnormal: subnormal values on every rank (a flush-to-zero build would lose them);
  * inf (one rank +-inf), inf_cancel (+inf and -inf: NaN), nan (one rank NaN), overflow (every rank 0.75 FLT_MAX: +-inf).

The lane assignment is a random permutation, except that lane n - 2 is always an order lane: it sits next to the vote in the
last, partial float4 of the bucket (n = n_params + 1 is 2 mod 4 for the policies of this project).
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np

SENTINEL_BITS = 0x7FBADBAD          # a NaN pattern: fills the memory around the bucket in the GPU tests
SPECIALS = ("neg_zero", "mixed_zero", "subnormal", "inf", "inf_cancel", "nan", "overflow")
F32_MAX = float(np.finfo(np.float32).max)


def rank_order_sum(g: np.ndarray) -> np.ndarray:
    """((g[0] + g[1]) + g[2]) + ... in FP32, element by element: the sum dn_ppo_allreduce promises on every rank."""
    g = np.asarray(g, dtype=np.float32)
    s = g[0].copy()
    with np.errstate(all="ignore"):
        for r in range(1, len(g)):
            s = s + g[r]
    return s


def reversed_sum(g: np.ndarray) -> np.ndarray:
    return rank_order_sum(np.asarray(g)[::-1])


def pairwise_sum(g: np.ndarray) -> np.ndarray:
    """sum(first half) + sum(second half), recursively (W = 3: g0 + (g1 + g2); W = 4: (g0 + g1) + (g2 + g3))."""
    g = np.asarray(g, dtype=np.float32)
    if len(g) == 1:
        return g[0].copy()
    h = len(g) // 2
    with np.errstate(all="ignore"):
        return pairwise_sum(g[:h]) + pairwise_sum(g[h:])


def rotated_sum(g: np.ndarray, start: int) -> np.ndarray:
    """Rank order starting at rank `start` (what a kernel that began its sum at its own rank would compute)."""
    g = np.asarray(g)
    return rank_order_sum(np.concatenate([g[start:], g[:start]]))


def _scaled(rng, shape, lo, hi):
    """+-(1 + u) 2^e with e uniform in lo..hi."""
    sign = np.where(rng.random(shape) < 0.5, -1.0, 1.0)
    return (sign * (1.0 + rng.random(shape)) * np.exp2(rng.integers(lo, hi + 1, shape))).astype(np.float32)


def _order_lanes(rng, count: int, world: int) -> np.ndarray:
    """[world, count] lanes whose rank-order sum differs from the reversed and the pairwise sums (W >= 3)."""
    out = np.zeros((world, 0), np.float32)
    while out.shape[1] < count:
        m = 4 * (count - out.shape[1]) + 64
        e0 = rng.integers(-10, 11, m)
        g = np.empty((world, m), np.float32)
        g[0] = _scaled(rng, m, 0, 0) * np.exp2(e0).astype(np.float32)
        for r in range(1, world):               # 1 .. 2^-26 of the first rank's magnitude: partial cancellation and lost bits
            g[r] = _scaled(rng, m, 0, 0) * np.exp2(e0 - rng.integers(0, 27, m)).astype(np.float32)
        flip = rng.random(m) < 0.5              # half the lanes: the last rank nearly cancels the first
        g[world - 1] = np.where(flip, -g[0] * np.float32(1.0 + 2.0 ** -20), g[world - 1])
        if world >= 3:
            ref = rank_order_sum(g).view(np.uint32)
            keep = (ref != reversed_sum(g).view(np.uint32)) & (ref != pairwise_sum(g).view(np.uint32))
            g = g[:, keep]
        out = np.concatenate([out, g], axis=1)
    return out[:, :count]


def make_inputs(n: int, world: int, seed: Tuple[int, ...]) -> Tuple[np.ndarray, Dict[str, np.ndarray]]:
    """([world, n] float32 buckets of every rank for one call, {category: lane indices}).  `seed` names the call (call index,
    handle); row r additionally depends on r, so no two ranks and no two calls share a bucket."""
    m = n - 1                                   # lanes before the vote
    joint = np.random.default_rng([*seed, world, n])
    perm = joint.permutation(m)
    n_order, n_special = m // 4, max(8, m // 64)
    lanes: Dict[str, np.ndarray] = {}
    pos = 0
    for cat, cnt in [("order", n_order)] + [(s, n_special) for s in SPECIALS]:
        lanes[cat] = perm[pos:pos + cnt]
        pos += cnt
    lanes["wide"] = perm[pos:]
    if m - 1 not in set(lanes["order"].tolist()):        # lane n - 2 is an order lane (moved there from wherever it was)
        for cat in lanes:
            lanes[cat] = lanes[cat][lanes[cat] != m - 1]
        lanes["order"] = np.append(lanes["order"], m - 1)
    g = np.empty((world, n), np.float32)
    for r in range(world):
        g[r] = _scaled(np.random.default_rng([*seed, world, n, 1000 + r]), n, -20, 20)
    W = world
    o = lanes["order"]
    g[:, o] = _order_lanes(joint, len(o), W)
    z = lanes["neg_zero"]
    g[:, z] = -0.0
    z = lanes["mixed_zero"]
    zs = np.where(joint.random((W, len(z))) < 0.5, -0.0, 0.0).astype(np.float32)
    zs[0] = -0.0
    zs[1 + joint.integers(0, W - 1, len(z)), np.arange(len(z))] = 0.0
    g[:, z] = zs
    s = lanes["subnormal"]
    bits = joint.integers(1, 1 << 21, (W, len(s)), dtype=np.uint32) | np.where(joint.random((W, len(s))) < 0.5, 0x80000000, 0).astype(np.uint32)
    g[:, s] = bits.view(np.float32)
    for cat in ("inf", "inf_cancel", "nan"):
        li = lanes[cat]
        who = joint.integers(0, W, len(li))
        if cat == "inf":
            g[who, li] = np.where(joint.random(len(li)) < 0.5, -np.inf, np.inf).astype(np.float32)
        elif cat == "nan":
            g[who, li] = (0x7FC00000 | joint.integers(1, 1 << 22, len(li), dtype=np.uint32)).view(np.float32)
        else:
            other = (who + 1 + joint.integers(0, W - 1, len(li))) % W
            g[who, li] = np.inf
            g[other, li] = -np.inf
    li = lanes["overflow"]
    g[:, li] = np.where(joint.random(len(li)) < 0.5, -0.75, 0.75).astype(np.float32) * np.float32(F32_MAX)
    g[:, n - 1] = (joint.random(W) < 0.5).astype(np.float32)            # the votes
    return g, lanes


def compare(got: np.ndarray, want: np.ndarray) -> Dict[str, int]:
    """Bit mismatches outside the NaN lanes of `want`, and lanes where exactly one of the two is NaN (NaN payloads are not
    compared), with the first offending index (-1: none)."""
    gn, wn = np.isnan(got), np.isnan(want)
    bits = ~wn & ~gn & (got.view(np.uint32) != want.view(np.uint32))
    bad = np.flatnonzero(bits | (gn != wn))
    return {"bit_mismatches": int(bits.sum()), "nan_mismatches": int((gn != wn).sum()), "first_bad": int(bad[0]) if len(bad) else -1}
