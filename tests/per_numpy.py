"""numpy restatement of prioritized replay (csrc/ring.cuh): the sum tree, the stratified draw, the importance weights and the
priorities, in the same Float32 / Float64 rounding order as the kernels."""
import ctypes as C

import numpy as np

STREAM_PER = 0x5052


def p2_of(cap):
    p = 1
    while p < cap:
        p <<= 1
    return p


def build_tree(leaves, cap):
    """leaves [cap] float32 by physical slot -> (tree [2 P2] float32, P2); every node RN32(left + right)"""
    p2 = p2_of(cap)
    t = np.zeros(2 * p2, np.float32)
    t[p2:p2 + cap] = np.asarray(leaves, np.float32)
    lo = p2
    while lo > 1:
        lo >>= 1
        t[lo:2 * lo] = t[2 * lo:4 * lo:2] + t[2 * lo + 1:4 * lo:2]
    return t, p2


def u53(O, seed, j, ctr, stream=STREAM_PER):
    w = (C.c_uint32 * 4)()
    O.lib().oracle_philox(int(seed) & (2**64 - 1), int(j), int(ctr), stream, w)
    return float(((w[0] >> 5) << 26) | (w[1] >> 6)) * (1.0 / 9007199254740992.0)


def draw(O, t, p2, seed, j, ctr, B):
    """row j of B of update ctr -> (physical slot, its leaf)"""
    x = np.float32((float(j) + u53(O, seed, j, ctr)) * float(t[1]) / float(B))
    n = 1
    while n < p2:
        L, R = t[2 * n], t[2 * n + 1]
        if x < L or R == 0:
            n = 2 * n
        else:
            x = np.float32(x - L)
            n = 2 * n + 1
    return n - p2, t[n]


def logical(slot, head, length, cap):
    return (slot - head + length) % cap


def weights(leaves, length, root, beta):
    """RN32(x_j^-beta / max_k x_k^-beta), x_j = leaf_j len / root in Float64"""
    raw = [(float(l) * float(length) / float(root)) ** (-float(beta)) for l in leaves]
    m = max(raw)
    return np.array([np.float32(r / m) for r in raw], np.float32)


def priority(y, q, alpha, eps):
    d = np.float32(np.float32(y) - np.float32(q))
    return np.float32((abs(float(d)) + float(np.float32(eps))) ** float(np.float32(alpha)))


def sample(O, leaves, cap, head, length, seed, B, beta, ctr=0):
    """what replay_sample_prioritized returns: (logical indices [B], weights [B], slots [B])"""
    t, p2 = build_tree(leaves, cap)
    slots, lv = zip(*[draw(O, t, p2, seed, j, ctr, B) for j in range(B)])
    idx = np.array([logical(s, head, length, cap) for s in slots], np.int32)
    return idx, weights(lv, length, t[1], beta), np.array(slots)
