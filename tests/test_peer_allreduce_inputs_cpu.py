"""The inputs and the rank-order reference of tests/test_gpu_ppo_peer_allreduce.py, without a GPU: they can tell summation
orders apart, and every special lane has the sum IEEE FP32 prescribes.  This is what makes the GPU test fail for a kernel that
sums in another order, flushes subnormals or loses a sign of zero, without building such a kernel."""
import numpy as np
import pytest

from tests import peer_allreduce_inputs as I

NS = (4234, 73610, 803594)          # n_params + 1 of the three policies the GPU test exchanges


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


@pytest.mark.parametrize("world", (2, 3, 4))
@pytest.mark.parametrize("n", NS)
def test_inputs_cover_every_category_and_are_reproducible(n, world):
    g, lanes = I.make_inputs(n, world, (5, 1))
    assert g.shape == (world, n) and g.dtype == np.float32
    every = np.concatenate(list(lanes.values()))
    assert len(every) == n - 1 and len(np.unique(every)) == n - 1          # every lane but the vote, once
    assert n - 2 in set(lanes["order"].tolist())                           # the partial float4 next to the vote
    assert all(len(lanes[c]) >= 8 for c in lanes) and len(lanes["order"]) >= (n - 1) // 4
    g2, lanes2 = I.make_inputs(n, world, (5, 1))
    assert np.array_equal(_bits(g), _bits(g2)) and all(np.array_equal(lanes[c], lanes2[c]) for c in lanes)
    other, _ = I.make_inputs(n, world, (6, 1))
    assert (_bits(g) != _bits(other)).mean() > 0.5                          # another call: another bucket
    for a in range(world):                                                  # and no two ranks send the same bucket
        for b in range(a):
            assert (_bits(g[a]) != _bits(g[b])).mean() > 0.5
    w = g[:, lanes["wide"]]
    e = np.log2(np.abs(w))
    assert e.min() >= -20 and e.max() <= 21 and e.min() < -19 and e.max() > 20
    assert set(np.unique(g[:, n - 1]).tolist()) <= {0.0, 1.0}


@pytest.mark.parametrize("world", (3, 4))
@pytest.mark.parametrize("n", NS)
def test_order_lanes_tell_summation_orders_apart(n, world):
    """Every order lane gives a different FP32 sum reversed and as a pairwise tree; starting the rank order at another rank
    changes a large share of them."""
    for call in range(3):
        g, lanes = I.make_inputs(n, world, (call, 0))
        o = lanes["order"]
        ref = _bits(I.rank_order_sum(g)[o])
        assert np.all(ref != _bits(I.reversed_sum(g)[o]))
        assert np.all(ref != _bits(I.pairwise_sum(g)[o]))
        for start in range(1, world):
            assert (ref != _bits(I.rotated_sum(g, start)[o])).mean() > 0.25, start
        assert np.all(np.isfinite(I.rank_order_sum(g)[o]))


@pytest.mark.parametrize("world", (2, 3, 4))
def test_rank_order_sum_of_the_special_lanes(world):
    n = 73610
    g, lanes = I.make_inputs(n, world, (1, 1))
    s = I.rank_order_sum(g)
    assert np.all(_bits(s[lanes["neg_zero"]]) == 0x80000000)              # -0 + -0 = -0
    assert np.all(_bits(s[lanes["mixed_zero"]]) == 0)                      # -0 + +0 = +0
    zs = g[:, lanes["mixed_zero"]]
    assert np.all(np.signbit(zs).any(0)) and np.all((~np.signbit(zs)).any(0))
    sub = g[:, lanes["subnormal"]]
    assert np.all((np.abs(sub) < 2.0 ** -126) & (sub != 0))
    ss = s[lanes["subnormal"]]
    exact = sub.astype(np.float64).sum(0)                                  # subnormal sums are exact in FP32
    assert np.array_equal(ss.astype(np.float64), exact)
    assert ((np.abs(ss) < 2.0 ** -126) & (ss != 0)).mean() > 0.3           # a flush-to-zero kernel would return 0 there
    assert np.all(np.isinf(s[lanes["inf"]]))
    gi = g[:, lanes["inf"]]
    assert np.array_equal(np.sign(s[lanes["inf"]]), np.sign(np.where(np.isinf(gi), gi, 0.0).sum(0)))
    assert np.all(np.isnan(s[lanes["inf_cancel"]])) and np.all(np.isnan(s[lanes["nan"]]))
    assert np.all(np.isinf(s[lanes["overflow"]]))
    assert np.all(np.isfinite(s[lanes["wide"]]))
    assert s[n - 1] == g[:, n - 1].sum() and float(s[n - 1]).is_integer()  # the vote: the exact count of voting ranks


def test_compare_ignores_nan_payloads_but_not_nan_positions_or_zero_signs():
    want = np.array([np.nan, 1.0, -0.0, np.inf], np.float32)
    got = want.copy()
    got[0] = np.array([0x7FC00123], np.uint32).view(np.float32)[0]
    assert I.compare(got, want) == {"bit_mismatches": 0, "nan_mismatches": 0, "first_bad": -1}
    got[2] = 0.0
    assert I.compare(got, want) == {"bit_mismatches": 1, "nan_mismatches": 0, "first_bad": 2}
    got[2], got[1] = -0.0, np.nan
    assert I.compare(got, want) == {"bit_mismatches": 0, "nan_mismatches": 1, "first_bad": 1}
