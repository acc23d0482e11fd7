"""numpy restatement of n-step returns (csrc/ring.cuh): the successor-link rule a write applies and the walk an n-step row takes, on
what replay_get returns (logical order, oldest first) and in the same Float32 / Float64 rounding order as the kernels."""
import numpy as np


def continues(S, S2, D, p, i):
    """does record i continue record p?  done(p) == 0 and s(i) == s'(p) in all 9 fields, bit for bit"""
    return D[p] == 0 and np.array_equal(S[:, i].view(np.uint32), S2[:, p].view(np.uint32))


def after_write(prev, len_before, S, S2, D, n_written, width, cap):
    """the links after a write of n_written records, `width` instances per step.  prev: the links [len_before] before it (logical
    indices, -1 none); S, S2, D: the memory after it (replay_get).  The surviving old records keep their links (shifted by the
    records the write pushed out); every new record i gets -1, and p = i - width gets i when p exists and i continues p."""
    n = S.shape[1]
    m = min(n_written, cap)
    old = n - m
    shift = len_before - old
    nx = np.full(n, -1, np.int32)
    for o in range(old):
        v = prev[o + shift]
        nx[o] = v - shift if v >= 0 else -1
    for i in range(old, n):
        p = i - width
        if p >= 0 and continues(S, S2, D, p, i):
            nx[p] = i
    return nx


class Ring:
    """a host replay memory of capacity cap that keeps its links by after_write: push(S, A, R, S2, D, width)"""

    def __init__(self, cap):
        self.cap = cap
        self.S, self.A, self.R, self.S2, self.D = (np.zeros((9, 0), np.float32), np.zeros((2, 0), np.float32), np.zeros(0, np.float32),
                                                   np.zeros((9, 0), np.float32), np.zeros(0, np.float32))
        self.next = np.zeros(0, np.int32)

    def push(self, S, A, R, S2, D, width):
        n0 = self.R.size
        keep = lambda x, y: np.concatenate([x, y], axis=-1)[..., -self.cap:]
        self.S, self.A, self.R, self.S2, self.D = (keep(self.S, S), keep(self.A, A), keep(self.R, R), keep(self.S2, S2), keep(self.D, D))
        self.next = after_write(self.next, n0, self.S, self.S2, self.D, R.size, width, self.cap)


def walk(R, D, nx, i0, n, gamma):
    """the chain from record i0: (last record, RN32(R), done folded with γ^{k-1}, k) — Python floats are Float64 and round each
    operation, as the kernel's __dmul_rn / __dadd_rn"""
    g = float(np.float32(gamma))
    gp, ret, k, last = 1.0, float(R[i0]), 1, i0
    while k < n and D[last] == 0 and nx[last] >= 0:
        last = int(nx[last])
        gp = gp * g
        ret = ret + gp * float(R[last])
        k += 1
    return last, np.float32(ret), np.float32(1.0 - gp * (1.0 - float(D[last]))), k


def sample(S, A, R, S2, D, nx, idx, n, gamma):
    """what replay_sample_nstep returns for the rows starting at the logical indices idx"""
    rows = [walk(R, D, nx, int(i), n, gamma) for i in idx]
    last = np.array([w[0] for w in rows])
    return (S[:, idx], A[:, idx], np.array([w[1] for w in rows], np.float32), S2[:, last], np.array([w[2] for w in rows], np.float32),
            np.array([w[3] for w in rows], np.int32))
