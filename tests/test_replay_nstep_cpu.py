"""n-step returns on the host: the successor-link rule of tests/nstep_numpy.py on hand-built write sequences, the walk at n = 1
against the 1-step row, and the bound on the discount the folded done gives the unchanged TD target."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import nstep_numpy as NN  # noqa: E402


def chain(states, done=None):
    """transitions of one instance through `states` [9][T+1]: (S, A, R, S2, D) of its T steps, r_t = t + 1"""
    T = states.shape[1] - 1
    D = np.zeros(T, np.float32) if done is None else np.asarray(done, np.float32)
    return (states[:, :T].copy(), np.zeros((2, T), np.float32), np.arange(1, T + 1, dtype=np.float32), states[:, 1:].copy(), D)


def interleave(chains):
    """one write of W = len(chains) instances per step: step t of instance i at position t * W + i"""
    W = len(chains)
    return [np.stack([c[f] for c in chains], axis=-1).reshape(c0.shape[:-1] + (-1,)) for f, c0 in enumerate(chains[0])], W


def states(rng, T):
    return rng.standard_normal((9, T + 1)).astype(np.float32)


def test_one_step_writes_link_a_chain():
    ring = NN.Ring(16)
    S, A, R, S2, D = chain(states(np.random.default_rng(0), 5))
    for t in range(5):
        ring.push(S[:, t:t + 1], A[:, t:t + 1], R[t:t + 1], S2[:, t:t + 1], D[t:t + 1], 1)
    np.testing.assert_array_equal(ring.next, [1, 2, 3, 4, -1])


def test_mixed_widths_resets_and_done():
    rng = np.random.default_rng(1)
    ring = NN.Ring(64)
    x0, x1 = states(rng, 3), states(rng, 3)
    (S, A, R, S2, D), W = interleave([chain(x0), chain(x1, done=[0, 0, 1])])   # a rollout-like write: 2 instances x 3 steps
    ring.push(S, A, R, S2, D, W)
    # positions: step t of instance i at 2t + i; instance 1's last step is terminal
    np.testing.assert_array_equal(ring.next, [2, 3, 4, 5, -1, -1])
    # one push of width 1 that continues instance 0 (p = 6 - 1 = 5 is instance 1's terminal step: no link), then one that
    # continues it again, then a reset
    y = np.concatenate([x0[:, 3:4], states(rng, 2)[:, :2]], axis=1)
    s, a, r, s2, d = chain(y)
    ring.push(s[:, :1], a[:, :1], r[:1], s2[:, :1], d[:1], 1)
    np.testing.assert_array_equal(ring.next, [2, 3, 4, 5, -1, -1, -1])
    ring.push(s[:, 1:2], a[:, 1:2], r[1:2], s2[:, 1:2], d[1:2], 1)
    np.testing.assert_array_equal(ring.next, [2, 3, 4, 5, -1, -1, 7, -1])
    z = states(rng, 1)   # a reset: its s equals nobody's s'
    ring.push(*chain(z), 1)
    np.testing.assert_array_equal(ring.next, [2, 3, 4, 5, -1, -1, 7, -1, -1])
    # a write of width 2 whose records do not continue the records 2 before them
    (S, A, R, S2, D), W = interleave([chain(states(rng, 1)), chain(states(rng, 1))])
    ring.push(S, A, R, S2, D, W)
    np.testing.assert_array_equal(ring.next, [2, 3, 4, 5, -1, -1, 7, -1, -1, -1, -1])


def test_write_larger_than_cap_and_wrap_around():
    rng = np.random.default_rng(2)
    ring = NN.Ring(4)
    ring.push(*chain(states(rng, 6)), 1)           # 6 records of one chain, width 1: the last 4 survive, linked
    np.testing.assert_array_equal(ring.next, [1, 2, 3, -1])
    ring = NN.Ring(5)
    x = states(rng, 7)
    S, A, R, S2, D = chain(x)
    ring.push(S[:, :3], A[:, :3], R[:3], S2[:, :3], D[:3], 1)
    for t in range(3, 7):                          # wraps: the oldest records leave, the links shift with them
        ring.push(S[:, t:t + 1], A[:, t:t + 1], R[t:t + 1], S2[:, t:t + 1], D[t:t + 1], 1)
    np.testing.assert_array_equal(ring.next, [1, 2, 3, 4, -1])
    np.testing.assert_array_equal(ring.R, [3, 4, 5, 6, 7])
    # a write of width 2 larger than the ring: only pairs inside the surviving records can link
    (S, A, R, S2, D), W = interleave([chain(states(rng, 4)), chain(states(rng, 4))])
    ring.push(S, A, R, S2, D, W)
    np.testing.assert_array_equal(ring.next, [2, 3, 4, -1, -1])


def test_k1_rows_equal_one_step_rows():
    rng = np.random.default_rng(3)
    ring = NN.Ring(50)
    S, A, R, S2, D = chain(states(rng, 40), done=(rng.uniform(size=40) < 0.2).astype(np.float32))
    R = rng.standard_normal(40).astype(np.float32)
    ring.push(S, A, R, S2, D, 1)
    idx = np.arange(40)
    for gamma in (0.0, 0.5, 0.99, 1.0):
        s, a, r, s2, d, k = NN.sample(ring.S, ring.A, ring.R, ring.S2, ring.D, ring.next, idx, 1, gamma)
        assert np.all(k == 1)
        for x, y in ((s, ring.S), (a, ring.A), (r, ring.R), (s2, ring.S2), (d, ring.D)):
            np.testing.assert_array_equal(x.view(np.uint32), y.view(np.uint32))
    # n > 1: a terminal record ends the walk, and done stays 1
    s, a, r, s2, d, k = NN.sample(ring.S, ring.A, ring.R, ring.S2, ring.D, ring.next, idx, 16, 0.9)
    term = np.flatnonzero(ring.D == 1)
    assert np.all(d[term] == 1) and np.all(k[term] == 1)


def test_fold_bound():
    """with done = 0 the epilogue's Float32 discount γ (1 - done_out) is γ^k to within 2^-23 (two ulps of 1): done_out =
    RN32(1 - γ^{k-1}) is off by at most 2^-25, 1 - done_out rounds once more and the product with γ once more"""
    worst = 0.0
    for gamma in np.linspace(0.0, 1.0, 201, dtype=np.float32).tolist() + [0.9, 0.95, 0.99, 0.995, 0.999, 1.0 - 2**-24]:
        g = np.float32(gamma)
        R = np.zeros(16, np.float32)
        D = np.zeros(16, np.float32)
        nx = np.append(np.arange(1, 16), -1).astype(np.int32)
        for n in range(1, 17):
            _, _, done_out, k = NN.walk(R, D, nx, 0, n, g)
            assert k == n
            disc = np.float32(g * np.float32(np.float32(1.0) - done_out))   # what y = r + (γ (1 - done)) q' multiplies q' by
            err = abs(float(disc) - float(g) ** k)
            worst = max(worst, err)
            assert err <= 2.0**-23, (float(g), k, err)
    assert worst > 0.0   # the fold is not exact everywhere: the bound is what holds
