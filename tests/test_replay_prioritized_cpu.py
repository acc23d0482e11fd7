"""Prioritized replay without a GPU: the numpy restatement's stratified sampler draws slot s with probability p_s / sum p, and the
drivers' β schedule runs from beta0 at the first episode to 1 at the last."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_weighted as OW  # noqa: E402
import per_numpy as PN  # noqa: E402


def test_stratified_sampler_matches_priorities(O):
    from scipy.stats import chisquare
    cap = 37                                            # not a power of two: padding leaves stay 0
    rng = np.random.default_rng(3)
    leaves = rng.uniform(0.05, 2.0, cap).astype(np.float32)
    leaves[[4, 11, 30]] = 0.0                           # never drawn
    t, p2 = PN.build_tree(leaves, cap)
    B, updates = 64, 300
    counts = np.zeros(cap)
    for u in range(updates):
        for j in range(B):
            s, leaf = PN.draw(O, t, p2, 99, j, u, B)
            assert s < cap and leaf > 0 and leaf == leaves[s]
            counts[s] += 1
    assert counts[[4, 11, 30]].sum() == 0
    keep = leaves > 0
    p = leaves[keep].astype(np.float64)
    expect = p / p.sum() * counts.sum()
    assert chisquare(counts[keep], expect).pvalue > 1e-3


def test_tree_is_a_function_of_its_leaves():
    leaves = np.array([1e8, 1.0, 3.0, 1e-7, 0.5], np.float32)   # sums that round in Float32
    t, p2 = PN.build_tree(leaves, 5)
    f = np.float32
    a, b, c = f(1e8) + f(1.0), f(3.0) + f(1e-7), f(0.5) + f(0.0)
    assert p2 == 8 and t[1] == (a + b) + (c + f(0.0))
    assert np.all(t[p2 + 5:] == 0)


def test_beta_schedule(sb):
    from shems_b200.ddpg import per_beta
    assert per_beta(0.4, 1, 50) == pytest.approx(0.4)
    assert per_beta(0.4, 50, 50) == 1.0
    vals = [per_beta(0.4, i, 50) for i in range(1, 51)]
    assert np.all(np.diff(vals) > 0)
    assert per_beta(0.4, 1, 1) == 1.0


def test_weighted_oracle(O, tmp_path):
    """the weighted oracle update is the oracle's update when every weight is 1, and differs from it otherwise"""
    WL = OW.load(str(tmp_path))
    kw = dict(batch=16, l1=12, l2=20)
    rng = np.random.default_rng(4)
    s, s2 = rng.uniform(-1, 3, (9, 16)).astype(np.float32), rng.uniform(-1, 3, (9, 16)).astype(np.float32)
    a, r = rng.uniform(-1, 1, (2, 16)).astype(np.float32), rng.uniform(-5, 1, 16).astype(np.float32)
    done = np.zeros(16, np.float32)
    nets = []
    for w in (None, np.ones(16, np.float32), rng.uniform(0.1, 1, 16).astype(np.float32)):
        orc = O.OracleDdpg(O.default_ddpg_params(**kw))
        orc.init(9)
        if w is None:
            orc.update_batch(s, a, r, s2, done)
        else:
            q, y = OW.update_batch_weighted(WL, orc, s, a, r, s2, done, w)
            assert q.shape == y.shape == (16,) and np.all(np.isfinite(q))
        nets.append([orc.get_grad(1, k)[0] for k in range(3)])
    for g0, g1, g2 in zip(*nets):
        np.testing.assert_array_equal(g0, g1)
        assert not np.array_equal(g0, g2)
