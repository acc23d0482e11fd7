"""Float64 restatement of the gradients of one replay() step (DDPG.jl:131-143), with a rigorous per-element error bound.

numpy float64 throughout; a net is [(W1, b1), (W2, b2), (W3, b3)] with W in the layout of Learner.get_layer / get_grad reshaped to
Wt[in][out] (Flux).  The formulas are those of oracle/ddpg_oracle.c and tests/test_oracle_ddpg.py:
  normalisation (s - lo) / ((hi - lo) + 1f-8) in Float32, TD target y = r + γ(1 - d) q', dq = 2(q - y)/B, the critic's backward
  pass, dqπ = -1/B, the dX chain through the critic into the action inputs times 1 - a², the actor's backward pass, both losses.
relu'(0) = 0 (Zygote's x > 0) everywhere.

critic_pass() and actor_pass() are separate: the actor's gradients are taken through the UPDATED critic (phase 2 of an update only
moves the targets), so a test can hand actor_pass() the critic the device holds after the step.

track=True adds a running error bound to every gradient: each product is bounded by
  |got - ref| <= |eA|·|B| + |A|·|eB| + |eA|·|eB| + eps_K · (|A| + eA)·(|B| + eB),   eps_K = U_TF32 + K · 2^-24,
the magnitude pass (the same chain on |W|, |x| and |upstream gradient|, with the reference's relu masks) carrying the operands'
own bounds.  U_TF32 = 2^-9 covers truncating or rounding both operands of a product to TF32 (10 explicit bits); K · 2^-24 covers
fp32 accumulation of K terms in any order or split.  The same eps is used for every product, so the bound holds whichever of the
fp32 SIMT or TF32 tensor-core kernels computed it.  A relu unit whose reference pre-activation lies within its own bound may flip
on the device: its full upstream |gradient| is added to the bound of what it feeds.
"""
import numpy as np

U_TF32 = 2.0 ** -9
U_FP32 = 2.0 ** -24
STATE = 9


def eps(K):
    return U_TF32 + K * U_FP32


def normalize(s, s_min, s_max):
    """[9][B] float32 states -> [B][9] float64 inputs, computed in Float32 as the device and the oracle do"""
    s = np.asarray(s, np.float32)
    lo, hi = np.asarray(s_min, np.float32), np.asarray(s_max, np.float32)
    den = (hi - lo) + np.float32(1e-8)
    return ((s - lo[:, None]) / den[:, None]).T.astype(np.float64)


def relu_mask(z):
    return (z > 0).astype(np.float64)


class Val:
    """a float64 value with an elementwise bound on the device's deviation from it (err is None: no bound tracked)"""

    def __init__(self, v, err=None):
        self.v, self.err = v, err


def _prod(A, B, K, track):
    """A @ B, and its bound when tracked (A, B: Val)"""
    v = A.v @ B.v
    if not track:
        return Val(v)
    aA, aB = np.abs(A.v), np.abs(B.v)
    eA = A.err if A.err is not None else np.zeros_like(aA)
    eB = B.err if B.err is not None else np.zeros_like(aB)
    if B.err is None:                     # exact operand (weights): two of the four products vanish
        return Val(v, eA @ aB + eps(K) * ((aA + eA) @ aB))
    e = eA @ aB + aA @ eB + eA @ eB + eps(K) * ((aA + eA) @ (aB + eB))
    return Val(v, e)


def _add_bias(z, b, K, track):
    v = z.v + b[None, :]
    if not track:
        return Val(v)
    return Val(v, z.err + eps(K) * np.abs(b)[None, :])


def _colsum(d, track):
    """sum over the batch of d [B][n] (a bias gradient)"""
    v = d.v.sum(0)
    if not track:
        return Val(v)
    B = d.v.shape[0]
    return Val(v, d.err.sum(0) + eps(B) * (np.abs(d.v) + d.err).sum(0))


def forward(net, x, track=False):
    """x: Val [B][in].  Returns the pre-activations z1, z2, z3 and activations h1, h2 (Val)."""
    (W1, b1), (W2, b2), (W3, b3) = net
    f = {"x": x}
    z1 = _add_bias(_prod(x, Val(W1), W1.shape[0], track), b1, W1.shape[0], track)
    h1 = Val(np.where(z1.v > 0, z1.v, 0.0), z1.err)           # relu is 1-Lipschitz: the bound carries over, flipped or not
    z2 = _add_bias(_prod(h1, Val(W2), W2.shape[0], track), b2, W2.shape[0], track)
    h2 = Val(np.where(z2.v > 0, z2.v, 0.0), z2.err)
    z3 = _add_bias(_prod(h2, Val(W3), W3.shape[0], track), b3, W3.shape[0], track)
    f.update(z1=z1, h1=h1, z2=z2, h2=h2, z3=z3)
    return f


def _mask(dh, z, track):
    """dz = dh · relu'(z); a unit whose pre-activation lies within its bound may flip and pass (or drop) all of dh"""
    m = relu_mask(z.v)
    v = dh.v * m
    if not track:
        return Val(v), None
    flip = np.abs(z.v) <= z.err
    e = dh.err * m + flip * (np.abs(dh.v) + dh.err)
    return Val(v, e), flip


def backward(net, f, dout, want_dx=False, track=False):
    """dout: Val [B][J] = d loss / d output.  Returns {grads: [(dW1, db1), (dW2, db2), (dW3, db3)] as Val, dz2, dz1, dx, flips}."""
    (W1, b1), (W2, b2), (W3, b3) = net
    B = dout.v.shape[0]
    T = lambda a: Val(a.v.T, None if a.err is None else a.err.T)
    dW3 = _prod(T(f["h2"]), dout, B, track)
    db3 = _colsum(dout, track)
    dh2 = _prod(dout, Val(W3.T), W3.shape[1], track)
    dz2, flip2 = _mask(dh2, f["z2"], track)
    dW2 = _prod(T(f["h1"]), dz2, B, track)
    db2 = _colsum(dz2, track)
    dh1 = _prod(dz2, Val(W2.T), W2.shape[1], track)
    dz1, flip1 = _mask(dh1, f["z1"], track)
    dW1 = _prod(T(f["x"]), dz1, B, track)
    db1 = _colsum(dz1, track)
    out = {"grads": [(dW1, db1), (dW2, db2), (dW3, db3)], "dh2": dh2, "dz2": dz2, "dh1": dh1, "dz1": dz1, "flips": (flip1, flip2)}
    if want_dx:
        out["dx"] = _prod(dz1, Val(W1.T), W1.shape[1], track)
    return out


def _tanh(z, track):
    v = np.tanh(z.v)
    if not track:
        return Val(v)
    return Val(v, z.err + 4 * U_FP32)   # tanh is 1-Lipschitz; tanhf is within a few ulp of |tanh| <= 1


def critic_pass(actor_t, critic, critic_t, s_min, s_max, s, a, r, s2, done=None, gamma=0.99, track=False):
    """the critic half of one update on the minibatch s [9][B], a [2][B], r [B], s2 [9][B], done [B]:
    returns the critic's gradients, the loss, and the intermediates (q, y, dq, forward / backward dicts)"""
    B = s.shape[1]
    sn, s2n = normalize(s, s_min, s_max), normalize(s2, s_min, s_max)
    ex = (lambda x: 2 * U_FP32 * np.abs(x)) if track else (lambda x: None)   # the device may divide by a rounded reciprocal
    ft = forward(actor_t, Val(s2n, ex(s2n)), track)
    at = _tanh(ft["z3"], track)
    xs2 = Val(np.hstack([s2n, at.v]), np.hstack([ex(s2n), at.err]) if track else None)
    fqt = forward(critic_t, xs2, track)
    xs = np.hstack([sn, np.asarray(a, np.float64).T])
    fc = forward(critic, Val(xs, np.hstack([ex(sn), np.zeros((B, 2))]) if track else None), track)
    nd = 1.0 - (np.zeros(B) if done is None else np.asarray(done, np.float64))
    qt, q = fqt["z3"], fc["z3"]
    y = np.asarray(r, np.float64) + gamma * nd * qt.v[:, 0]
    dq = Val((2.0 * (q.v[:, 0] - y) / B)[:, None])
    if track:
        ey = gamma * nd * qt.err[:, 0] + 2 * U_FP32 * (np.abs(y) + gamma * np.abs(qt.v[:, 0]))
        dq.err = (2.0 / B * (q.err[:, 0] + ey) + 2 * U_FP32 * np.abs(dq.v[:, 0]))[:, None]
    bc = backward(critic, fc, dq, track=track)
    loss = float(np.mean((q.v[:, 0] - y) ** 2))
    return {"grads": bc["grads"], "loss": loss, "q": q.v[:, 0], "y": y, "dq": dq.v[:, 0], "fwd": fc, "bwd": bc, "xs": xs, "sn": sn}


def actor_pass(actor, critic, s_min, s_max, s, track=False):
    """the actor half: loss = -mean(critic(vcat(s_n, actor(s_n)))) through `critic` (the updated critic)"""
    B = s.shape[1]
    sn = normalize(s, s_min, s_max)
    ex = 2 * U_FP32 * np.abs(sn) if track else None
    fa = forward(actor, Val(sn, ex), track)
    api = _tanh(fa["z3"], track)
    xspi = Val(np.hstack([sn, api.v]), np.hstack([ex, api.err]) if track else None)
    fp = forward(critic, xspi, track)
    dqpi = Val(np.full((B, 1), -1.0 / B), np.zeros((B, 1)) if track else None)
    bp = backward(critic, fp, dqpi, want_dx=True, track=track)
    dxa = Val(bp["dx"].v[:, STATE:], None if not track else bp["dx"].err[:, STATE:])
    g = 1.0 - api.v ** 2
    dA = Val(dxa.v * g)
    if track:
        eg = 2 * np.abs(api.v) * api.err + api.err ** 2 + 2 * U_FP32
        dA.err = dxa.err * np.abs(g) + (np.abs(dxa.v) + dxa.err) * eg + 2 * U_FP32 * np.abs(dA.v)
    ba = backward(actor, fa, dA, track=track)
    loss = float(-np.mean(fp["z3"].v[:, 0]))
    return {"grads": ba["grads"], "loss": loss, "api": api.v, "dA": dA.v, "qpi": fp["z3"].v[:, 0], "fwd_actor": fa, "fwd_critic": fp,
            "bwd_critic": bp, "bwd_actor": ba, "xspi": xspi.v}
